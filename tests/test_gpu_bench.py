"""bench.py --dump-outputs on the device: what measure() gathers after its timed steps is x, g and f of that iterate,
at the sampled indices, as a separate solve of the same problem stepped to the same iteration has them."""
import numpy as np
import pytest

import bench

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("kind,dtype,l_odd", [("rosenbrock", "float64", bench.L_ODD), ("quadratic", "float64", bench.L_ODD),
                                              ("driver3_f32", "float32", 1.0)])
def test_dumped_outputs_are_the_last_timed_iterate(kind, dtype, l_odd, monkeypatch):
    import torch
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 1000)
    n, m, W, K = 20011, 5, 6, 3
    cx = bench.Ctx()
    r = bench.measure(cx, kind, n, m, dtype, l_odd, W, K, want_clocks=False, want_outputs=True)
    out = r["outputs"]
    idx = bench.dump_index(n)
    assert idx.size == 1000
    assert np.array_equal(out["index"], idx.astype(np.float64))

    ds = bench.DeviceSolve(cx, kind, n, m, dtype, l_odd, sharded_run=False)
    with torch.cuda.stream(cx.stream):
        assert ds.step_to(r["warmup_effective"] + K)
    torch.cuda.synchronize()
    for name in ("x", "g"):
        full = getattr(ds, name).cpu().numpy()
        assert out[name].dtype == np.dtype(dtype)
        assert np.array_equal(out[name], full[idx]), name
    assert out["f"].dtype == np.dtype(dtype) and out["f"][0] == ds.prob.f[0]
    ds.close()
