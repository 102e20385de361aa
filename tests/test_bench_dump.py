"""bench.py --dump-outputs on the benchmark workloads' real plans (a stand-in model serves the tensors, no GPU): every parameter
and optimizer slot is written, MLP tensors whole, the directory stays under 64 MB, and the sampled rows are the same run to run."""
import os

import numpy as np
import pytest

import bench


class TensorSource(object):
    """The tensor-reading part of WideDeepModel: every element of a row holds the row's index (exact in float32 below 2^24)."""

    def __init__(self, plan):
        self.plan = plan

    def tensor_names(self):
        return list(self.plan.tensor_names)

    def n_slots(self, name):
        o = self.plan.lin_opt if name.startswith("linear/") else self.plan.dnn_opt
        return {"sgd": 0, "adagrad": 1, "ftrl": 2, "adam": 2, "rmsprop": 2}[o["kind"]]

    def get_tensor(self, name, slot=0):
        shape = self.plan.local_shape(name)
        rows = np.arange(shape[0], dtype=np.float32)
        return np.broadcast_to(rows.reshape((-1,) + (1,) * (len(shape) - 1)), shape)


@pytest.mark.parametrize("workload", ["criteo", "multihot", "wide"])
def test_dump_outputs_budget_and_fixed_sample(workload, tmp_path):
    from wide_deep_b200.plan import T_DENSE
    wl = bench.Workload(workload, 1)
    src = TensorSource(wl.plan(wl.batch, "bf16x3"))
    for d in ("a", "b"):
        bench.dump_outputs(src, 0.5, str(tmp_path / d))
    files = sorted(os.listdir(str(tmp_path / "a")))
    assert files == sorted(os.listdir(str(tmp_path / "b")))
    assert sum(os.path.getsize(str(tmp_path / "a" / f)) for f in files) <= 64 * 10 ** 6
    assert np.load(str(tmp_path / "a" / "loss.npy")).tolist() == [0.5]
    for name in src.tensor_names():
        for s in range(src.n_slots(name) + 1):
            f = name.replace("/", ".") + (".slot%d" % s if s else "") + ".npy"
            a, b = np.load(str(tmp_path / "a" / f)), np.load(str(tmp_path / "b" / f))
            assert a.dtype == np.float32 and np.array_equal(a, b), f
            full = src.get_tensor(name, s)
            assert a.shape[1:] == full.shape[1:] and 0 < a.shape[0] <= full.shape[0], f
            if src.plan.tensor_names[name][0] == T_DENSE:
                assert np.array_equal(a, full), f
            rows = a.reshape(a.shape[0], -1)[:, 0]                    # the rows kept, in order, each one intact
            assert np.all(np.diff(rows) > 0) and np.array_equal(a, full[rows.astype(np.int64)]), f
