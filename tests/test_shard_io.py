"""Shard I/O of PartialFC (partial_fc.py:38-60 resume, :71-87 save_params / save_FC / update_FC / update_from_tensor):
file names, file contents, resume fall-backs and the sub_weight aliasing, on CPU through the host-logic provider
(tests/oracle_ops.py) and on the GPU through the real kernels."""
import os
import shutil
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
GOLDEN_FILES = ("rank:0_softmax_weight.pt", "rank:0_softmax_weight_mom.pt", "FC_rank_0.pth")


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    g.build()
    import fedfr_b200
    return fedfr_b200


def _head(pkg, prefix, resume=False, rank=0, world=1, classes=300, sr=1.0, emb=64, batch=32, cpu=True, local_rank=0):
    kw = {}
    if cpu:
        from oracle_ops import OracleOps
        kw["_ops"] = OracleOps()
    return pkg.PartialFC(rank, local_rank, world, batch, resume, pkg.CosFace(s=64.0, m=0.4), classes, sample_rate=sr,
                         embedding_size=emb, prefix=str(prefix), **kw)


def _train_one_step(head, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.nn.functional.normalize(torch.randn(head.batch_size, head.embedding_size, generator=g)).to(head.device)
    y = torch.randint(0, head.num_classes, (head.batch_size,), generator=g).to(head.device)
    opt = torch.optim.SGD([{"params": head.parameters()}], lr=0.1, momentum=0.9, weight_decay=5e-4)
    x_grad, loss = head.forward_backward(y, x, opt)
    opt.step()
    head.update()
    opt.zero_grad(set_to_none=True)                  # the reference accumulates into sub_weight.grad across calls
    return x, y, x_grad, loss


def test_names_and_geometry(pkg, tmp_path):
    h = _head(pkg, tmp_path, rank=1, world=3, classes=1001, local_rank=1)
    assert (h.num_local, h.class_start, h.num_sample) == (334, 334, 334)           # partial_fc.py:34-36
    assert h.weight_name == os.path.join(str(tmp_path), "rank:1_softmax_weight.pt")            # partial_fc.py:38
    assert h.weight_mom_name == os.path.join(str(tmp_path), "rank:1_softmax_weight_mom.pt")    # partial_fc.py:39
    assert tuple(h.weight.shape) == (334, 64) and h.weight.dtype == torch.float32
    assert float(h.weight_mom.abs().max()) == 0.0 and 0.008 < float(h.weight.std()) < 0.012    # N(0, 0.01), zeros
    assert [p.data_ptr() for p in h.parameters()] == [h.weight.data_ptr()]         # sub_weight IS the shard at sr == 1
    assert list(h.state_dict().keys()) == ["sub_weight"] and h.update() == 0


@pytest.mark.parametrize("sr", [1.0, 0.5])
def test_save_params_resume_roundtrip(pkg, tmp_path, sr):
    a = _head(pkg, tmp_path, sr=sr)
    _train_one_step(a)
    assert float(a.weight_mom.abs().max()) > 0
    a.save_params()
    assert sorted(os.listdir(tmp_path)) == ["rank:0_softmax_weight.pt", "rank:0_softmax_weight_mom.pt"]
    on_disk = torch.load(a.weight_name)                                              # what the reference's ctor does (:43)
    assert isinstance(on_disk, torch.Tensor) and on_disk.dtype == torch.float32 and tuple(on_disk.shape) == (300, 64)
    b = _head(pkg, tmp_path, resume=True, sr=sr)
    assert torch.equal(b.weight, a.weight) and torch.equal(b.weight_mom, a.weight_mom)
    if sr == 1.0:
        assert b.sub_weight.data_ptr() == b.weight.data_ptr() and b.sub_weight_mom.data_ptr() == b.weight_mom.data_ptr()
    else:
        assert b.sub_weight.numel() == 0 and b.index is None                         # partial_fc.py:69
    # the resumed head continues exactly where the saved one would
    torch.manual_seed(5)
    ra = _train_one_step(a, seed=1)
    torch.manual_seed(5)
    rb = _train_one_step(b, seed=1)
    assert torch.equal(ra[2], rb[2]) and float(ra[3]) == float(rb[3]) and torch.equal(a.weight, b.weight)


def test_resume_without_files_reinitialises(pkg, tmp_path):
    h = _head(pkg, tmp_path, resume=True)                                            # partial_fc.py:45-47,52-54
    assert tuple(h.weight.shape) == (300, 64) and 0.008 < float(h.weight.std()) < 0.012
    assert float(h.weight_mom.abs().max()) == 0.0
    a = _head(pkg, tmp_path)
    torch.save(a.weight.data, a.weight_name)                                         # weight present, momentum missing
    h = _head(pkg, tmp_path, resume=True)
    assert torch.equal(h.weight, a.weight) and float(h.weight_mom.abs().max()) == 0.0


def test_save_FC_update_FC(pkg, tmp_path, capsys):
    a = _head(pkg, tmp_path, local_rank=0)
    a.save_FC()
    path = os.path.join(str(tmp_path), "FC_rank_0.pth")                              # partial_fc.py:76
    assert os.path.exists(path)
    b = _head(pkg, tmp_path)
    old_param, mom_before = b.sub_weight, b.weight_mom.clone()
    assert not torch.equal(a.weight, b.weight)
    b.update_FC()
    assert "Load weight from %s" % path in capsys.readouterr().out                   # partial_fc.py:84
    assert torch.equal(b.weight, a.weight) and torch.equal(b.weight_mom, mom_before)  # momentum is not touched
    assert b.sub_weight is not old_param and b.sub_weight.data_ptr() == b.weight.data_ptr()
    assert b.sub_weight.requires_grad and b.sub_weight.grad is None
    ra, rb = _train_one_step(a, seed=2), _train_one_step(b, seed=2)                  # and the loaded shard is the one used
    assert float(ra[3]) == float(rb[3]) and torch.equal(ra[2], rb[2])


def test_update_from_tensor(pkg, tmp_path):
    from oracle import partial_fc_oracle as O
    h = _head(pkg, tmp_path)
    new_w = torch.randn(300, 64, generator=torch.Generator().manual_seed(9)) * 0.05
    h.update_from_tensor(new_w.clone())              # partial_fc.py:85-87 (.to() of a same-device tensor aliases it)
    assert torch.equal(h.weight, new_w) and h.sub_weight.data_ptr() == h.weight.data_ptr()
    x, y, x_grad, loss = _train_one_step(h, seed=3)
    ref = O.forward_backward([x], [y], [new_w], 300, 64.0, 0.4)
    assert abs(float(loss) - float(ref.loss)) < 1e-4 * abs(float(ref.loss))
    assert float((x_grad - ref.x_grad[0]).abs().max()) < 1e-5


def test_files_interchange_with_reference_class(pkg, tmp_path):
    """The files the unmodified reference methods wrote (save_params / save_FC, tests/golden/make_golden_shard_io.py): this
    package resumes from them and loads them with update_FC, and the files it writes load back with plain torch.load."""
    for f in GOLDEN_FILES:
        shutil.copyfile(os.path.join(HERE, "golden", "shard_io", f), os.path.join(str(tmp_path), f))
    g = torch.Generator().manual_seed(4)                            # the tensors the reference saved
    w = torch.randn(300, 64, generator=g) * 0.01
    mom = torch.randn(300, 64, generator=g) * 0.001
    h = _head(pkg, tmp_path, resume=True)
    assert h.weight_name == os.path.join(str(tmp_path), GOLDEN_FILES[0]) and h.weight_mom_name == os.path.join(str(tmp_path), GOLDEN_FILES[1])
    assert torch.equal(h.weight, w) and torch.equal(h.weight_mom, mom)
    h2 = _head(pkg, tmp_path)
    h2.update_FC()
    assert torch.equal(h2.weight, w)
    _train_one_step(h)
    h.save_params()                                                 # ... and back: what partial_fc.py:43,50 would load
    assert torch.equal(torch.load(h.weight_name), h.weight) and torch.equal(torch.load(h.weight_mom_name), h.weight_mom)


@pytest.mark.gpu
@pytest.mark.parametrize("sr", [1.0, 0.5])
def test_gpu_checkpoint_roundtrip_and_loaders(pkg, tmp_path, sr):
    from oracle import partial_fc_oracle as O
    a = _head(pkg, tmp_path, sr=sr, emb=128, cpu=False)
    _train_one_step(a)
    torch.cuda.synchronize()
    a.save_params()
    a.save_FC()
    b = _head(pkg, tmp_path, resume=True, sr=sr, emb=128, cpu=False)
    assert b.weight.is_cuda and torch.equal(b.weight, a.weight) and torch.equal(b.weight_mom, a.weight_mom)
    c = _head(pkg, tmp_path, sr=sr, emb=128, cpu=False)
    c.update_FC()
    assert torch.equal(c.weight, a.weight) and c.sub_weight.data_ptr() == c.weight.data_ptr()
    if sr == 1.0:                                                 # the loaded shard is what the next step trains on
        new_w = torch.randn(300, 128, generator=torch.Generator().manual_seed(9)) * 0.05
        c.update_from_tensor(new_w)
        x, y, x_grad, loss = _train_one_step(c, seed=3)
        ref = O.forward_backward([x.cpu()], [y.cpu()], [new_w], 300, 64.0, 0.4)
        # which shard was used, not kernel numerics (those are test_gpu_parity's job): a stale shard is off by O(1)
        assert abs(float(loss) - float(ref.loss)) < 5e-2 * abs(float(ref.loss))
        assert float((x_grad.cpu() - ref.x_grad[0]).norm() / ref.x_grad[0].norm()) < 5e-2
