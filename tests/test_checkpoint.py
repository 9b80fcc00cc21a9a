"""Bridge-only checkpoint IO (SURVEY.md 8b on-disk contract, 8f rank 4): the two reference file formats
round-trip, files are exchangeable with the reference module in both directions, only rank 0 writes
under data parallelism. Host-side logic: runs without a GPU (the flat-arena snapshot path is covered by
the `gpu` test at the bottom)."""
import os
import pathlib
import sys

import numpy as np
import pytest
import torch

from oracle import bridge_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "tiny_bridge.npz")
TINY = dict(vision_dim=32, language_dim=64, num_blocks=2, num_heads_cross=2, num_heads_self=1)


def _bridge(seed=0):
    from vlm_bridge_b200 import BridgeLite

    torch.manual_seed(seed)
    return BridgeLite(dropout=0.1, **TINY)


def _fake_grads(m, seed):
    g = torch.Generator().manual_seed(seed)
    for p in m.parameters():
        p.grad = torch.randn(p.shape, generator=g) * 1e-2


def test_format_b_round_trip_and_file_set(tmp_path):
    from vlm_bridge_b200 import checkpoint as ck

    m = _bridge(0)
    opt = torch.optim.AdamW(m.parameters(), lr=1e-5, weight_decay=0.01)
    sched = torch.optim.lr_scheduler.CosineAnnealingLR(opt, T_max=10, eta_min=1e-6)
    for s in range(2):
        _fake_grads(m, s)
        opt.step()
        sched.step()
    w = ck.save_checkpoint(str(tmp_path), m, opt, epoch=3, best_val_loss=1.25, config={"learning_rate": 1e-5},
                           scheduler=sched, early_stopping_counter=2, is_best=True)
    w.wait()
    assert sorted(os.listdir(tmp_path)) == ["best_model.pth", "best_model_weights_only.pth", "latest_checkpoint.pth"]
    raw = torch.load(tmp_path / "latest_checkpoint.pth", weights_only=True)
    assert raw["epoch"] == 4 and raw["early_stopping_counter"] == 2            # training_orchestrator.py:114,134
    assert list(raw["model_state_dict"]) == ["bridge_module." + n for n in O.param_names(2)]
    assert all(v.dtype == torch.float32 for v in raw["model_state_dict"].values())
    assert set(torch.load(tmp_path / "best_model_weights_only.pth", weights_only=True)) == {"model_state_dict", "config"}

    m2 = _bridge(1)
    opt2 = torch.optim.AdamW(m2.parameters(), lr=1e-3)
    sched2 = torch.optim.lr_scheduler.CosineAnnealingLR(opt2, T_max=10, eta_min=1e-6)
    meta = ck.load_checkpoint(str(tmp_path / "best_model.pth"), m2, opt2, scheduler=sched2)
    assert meta == {"start_epoch": 4, "best_val_loss": 1.25, "early_stopping_counter": 2, "config": {"learning_rate": 1e-5}}
    for (n, a), (_, b) in zip(m.state_dict().items(), m2.state_dict().items()):
        assert torch.equal(a, b), n
    assert opt2.param_groups[0]["lr"] == opt.param_groups[0]["lr"]
    # resumed training continues identically
    _fake_grads(m, 9), _fake_grads(m2, 9)
    opt.step(), opt2.step()
    for a, b in zip(m.parameters(), m2.parameters()):
        assert torch.equal(a, b)


def test_format_a_and_cross_format_loading(tmp_path):
    from vlm_bridge_b200 import checkpoint as ck

    m = _bridge(2)
    ck.save_model(str(tmp_path / "a.pth"), m, {"vision_dim": 32, "language_dim": 64})
    raw = torch.load(tmp_path / "a.pth", weights_only=True)
    assert set(raw) == {"bridge_module_state_dict", "model_config"}            # full_model.py:450-461
    assert list(raw["bridge_module_state_dict"]) == O.param_names(2)
    ck.save_checkpoint(str(tmp_path), m, None, epoch=0, asynchronous=False)
    for f in ("a.pth", "latest_checkpoint.pth"):                               # either format into either loader
        for loader in (ck.load_model, lambda p, b: ck.load_checkpoint(p, b)):
            m2 = _bridge(3)
            loader(str(tmp_path / f), m2)
            assert all(torch.equal(a, b) for a, b in zip(m.parameters(), m2.parameters()))
    with pytest.raises(KeyError):
        torch.save({"something": 1}, tmp_path / "junk.pth")
        ck.load_model(str(tmp_path / "junk.pth"), m)
    bad = dict(raw["bridge_module_state_dict"])
    bad.pop("bridge_blocks.0.ln_cross.weight")
    torch.save({"bridge_module_state_dict": bad}, tmp_path / "short.pth")
    with pytest.raises(RuntimeError):                                          # strict, as the reference
        ck.load_model(str(tmp_path / "short.pth"), m)


def test_untrusted_pickles_are_refused_unless_asked(tmp_path):
    from vlm_bridge_b200 import checkpoint as ck

    m = _bridge(4)
    # the reference stores config.__dict__, which can hold arbitrary objects (training_orchestrator.py:124)
    ck.save_checkpoint(str(tmp_path), m, None, epoch=0, config={"checkpoint_dir": pathlib.Path("x")}, asynchronous=False)
    with pytest.raises(RuntimeError, match="trusted=True"):
        ck.load_checkpoint(str(tmp_path / "latest_checkpoint.pth"), _bridge(5))
    meta = ck.load_checkpoint(str(tmp_path / "latest_checkpoint.pth"), _bridge(5), trusted=True)
    assert meta["config"]["checkpoint_dir"] == pathlib.Path("x")
    assert not [f for f in os.listdir(tmp_path) if ".tmp." in f]               # atomic rename, nothing left behind


def _reference_bridge():
    """The reference `BridgeLite` at the TINY widths as its checkpoint files see it: the reference module's own
    state_dict, stored in tests/golden/tiny_bridge.npz by make_golden.py, as parameters under the same names, in
    the same registration order and with the same shapes."""
    z = np.load(GOLDEN)
    bridge = torch.nn.Module()
    for key in z.files:
        if not key.startswith("param/"):
            continue
        *path, leaf = key[len("param/"):].split(".")
        mod = bridge
        for part in path:
            if part not in mod._modules:
                mod.add_module(part, torch.nn.Module())
            mod = mod._modules[part]
        mod.register_parameter(leaf, torch.nn.Parameter(torch.from_numpy(z[key])))
    assert list(bridge.state_dict()) == O.param_names(2)
    return bridge


def test_files_are_exchangeable_with_the_reference_module(tmp_path):
    from vlm_bridge_b200 import checkpoint as ck

    class FullModelLike(torch.nn.Module):                                      # the prefix FullModel gives (full_model.py:68)
        def __init__(self, bridge):
            super().__init__()
            self.bridge_module = bridge

    ref = _reference_bridge()
    # reference -> here, Format A (FullModel.save_model) and Format B (save_checkpoint)
    torch.save({"bridge_module_state_dict": ref.state_dict(), "model_config": {}}, tmp_path / "ref_a.pth")
    ref_opt = torch.optim.AdamW(ref.parameters(), lr=1e-5, weight_decay=0.01)
    _fake_grads(ref, 1)
    ref_opt.step()
    full = FullModelLike(ref)
    torch.save({"epoch": 2, "model_state_dict": {k: v for k, v in full.state_dict().items() if "bridge_module" in k},
                "optimizer_state_dict": ref_opt.state_dict(), "best_val_loss": 0.5, "config": {},
                "early_stopping_counter": 0}, tmp_path / "ref_b.pth")
    mine = _bridge(8)
    ck.load_model(str(tmp_path / "ref_a.pth"), _bridge(8))
    opt = torch.optim.AdamW(mine.parameters(), lr=1e-5, weight_decay=0.01)
    assert ck.load_checkpoint(str(tmp_path / "ref_b.pth"), mine, opt)["start_epoch"] == 2
    assert all(torch.equal(a, b) for a, b in zip(ref.parameters(), mine.parameters()))
    # here -> reference: the reference's own load logic (training_orchestrator.py:166-176, full_model.py:471-472)
    _fake_grads(mine, 2)
    opt.step()
    ck.save_checkpoint(str(tmp_path), mine, opt, epoch=5, is_best=True, asynchronous=False)
    ckpt = torch.load(tmp_path / "latest_checkpoint.pth")
    ref2 = FullModelLike(_reference_bridge())
    msd = ref2.state_dict()
    for k, v in ckpt["model_state_dict"].items():
        assert k in msd
        msd[k] = v
    ref2.load_state_dict(msd)
    ref_opt2 = torch.optim.AdamW(ref2.parameters(), lr=1e-5, weight_decay=0.01)
    ref_opt2.load_state_dict(ckpt["optimizer_state_dict"])
    assert all(torch.equal(a, b) for a, b in zip(ref2.bridge_module.parameters(), mine.parameters()))
    ck.save_model(str(tmp_path / "mine_a.pth"), mine)
    ref2.bridge_module.load_state_dict(torch.load(tmp_path / "mine_a.pth")["bridge_module_state_dict"])


def _rank_worker(rank, world, port, base):
    import torch.distributed as dist

    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from vlm_bridge_b200 import checkpoint as ck

    w = ck.save_checkpoint(os.path.join(base, f"rank{rank}"), _bridge(0), None, epoch=0)
    assert (w is None) == (rank != 0)
    if w is not None:
        w.wait()
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(120)
def test_only_rank0_writes_world2(tmp_path):
    import socket

    import torch.multiprocessing as mp

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_rank_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert os.listdir(tmp_path / "rank0") == ["latest_checkpoint.pth"]
    assert not (tmp_path / "rank1").exists()


@pytest.mark.gpu
def test_flat_arena_snapshot_is_async_and_resumes_bit_exact(tmp_path):
    """On the GPU the snapshot is one D2H copy per arena (parameters, exp_avg, exp_avg_sq) enqueued on the
    stream; an optimizer step issued right after `save_checkpoint` returns must not leak into the file."""
    from vlm_bridge_b200 import BridgeAdamW, BridgeLite
    from vlm_bridge_b200 import checkpoint as ck

    cfg = dict(vision_dim=64, language_dim=128, num_blocks=2, num_heads_cross=2, num_heads_self=1)
    g = torch.Generator().manual_seed(3)
    vision, text = torch.randn(2, 9, 64, generator=g).cuda(), torch.randn(2, 6, 128, generator=g).cuda()

    def step(m, opt):
        opt.zero_grad(set_to_none=True)
        m(vision, text).float().square().mean().backward()
        opt.step()

    torch.manual_seed(0)
    m = BridgeLite(dropout=0.0, **cfg).cuda().train()
    opt = BridgeAdamW(m, lr=1e-3, weight_decay=0.01, max_grad_norm=0.3)
    step(m, opt), step(m, opt)
    want = {k: v.clone() for k, v in m.state_dict().items()}
    w = ck.save_checkpoint(str(tmp_path), m, opt, epoch=0, is_best=True)
    step(m, opt)                                           # races with the background writer on purpose
    after3 = {k: v.clone() for k, v in m.state_dict().items()}
    w.wait()
    torch.manual_seed(1)
    m2 = BridgeLite(dropout=0.0, **cfg).cuda().train()
    opt2 = BridgeAdamW(m2, lr=1e-3, weight_decay=0.01, max_grad_norm=0.3)
    meta = ck.load_checkpoint(str(tmp_path / "latest_checkpoint.pth"), m2, opt2)
    assert meta["start_epoch"] == 1
    for k, v in m2.state_dict().items():
        assert torch.equal(v, want[k]), k                  # the state at the time of the call, not later
    step(m2, opt2)                                         # third step from the restored state
    for k, v in m2.state_dict().items():
        assert torch.equal(v, after3[k]), k
    raw = torch.load(tmp_path / "best_model_weights_only.pth", weights_only=True)
    assert list(raw["model_state_dict"]) == ["bridge_module." + n for n in O.param_names(2)]
