"""CPU: `bench.py --dump-outputs` -- the loss, prediction and parameter gradients of a step as float32 .npy files, arrays
above their cap as the same seeded sample in every run."""
import numpy as np
import pytest
import torch

import bench


def _step():
    torch.manual_seed(0)
    model = torch.nn.Sequential(torch.nn.Linear(40, 30), torch.nn.Linear(30, 5))
    pred = model(torch.randn(8, 40))
    loss = pred.square().sum()
    loss.backward()
    return loss, pred, model


def test_dump_outputs_writes_fixed_samples(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_GRAD_ELEMS", 200)
    monkeypatch.setattr(bench, "DUMP_PRED_ELEMS", 16)
    loss, pred, model = _step()
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), loss, pred, model)
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == sorted(["loss.npy", "pred.npy"] + [f"grad.{k}.npy" for k, _ in model.named_parameters()])
    for name in names:
        a, b = np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)
        assert a.dtype == np.float32 and np.array_equal(a, b), name
    assert np.load(tmp_path / "a" / "loss.npy") == np.float32(loss.item())
    assert np.array_equal(np.load(tmp_path / "a" / "grad.1.weight.npy"), model[1].weight.grad.numpy())   # 150 <= cap: whole
    for name, t, cap in (("grad.0.weight", model[0].weight.grad, 200), ("pred", pred.detach(), 16)):
        idx = torch.randint(0, t.numel(), (cap,), generator=torch.Generator().manual_seed(t.numel())).sort().values
        assert np.array_equal(np.load(tmp_path / "a" / f"{name}.npy"), t.reshape(-1)[idx].numpy()), name


def test_dump_outputs_stays_within_its_budget(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 1000)
    with pytest.raises(AssertionError, match="exceeds"):
        bench.dump_outputs(str(tmp_path), *_step())
    assert not (tmp_path / "loss.npy").exists()


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "d"],
                                  ["--sweep", "attn", "--dump-outputs", "d"], ["--profile-step", "--dump-outputs", "d"]])
def test_bench_rejects_arguments_it_cannot_honour(argv, monkeypatch):
    monkeypatch.setattr("sys.argv", ["bench.py", *argv])
    with pytest.raises(SystemExit) as e:
        bench.main()
    assert e.value.code == 2
