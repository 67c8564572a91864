"""bench.py --dump-outputs and --steps: the writer, the CPU reference arm and the GPU arm."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import ROOT, orc

sys.path.insert(0, ROOT)
import bench  # noqa: E402


def run_bench(*args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_dump_outputs_writes_float32_and_samples_the_same_rows(tmp_path):
    # every row holds its own index, so a sampled row says where it came from
    rows = torch.arange(64, dtype=torch.float32)[:, None]
    outs = [("qkv", rows.expand(64, 40).to(torch.bfloat16)), ("o", rows.expand(64, 24).to(torch.bfloat16))]
    bench.dump_outputs(str(tmp_path / "all"), outs)
    for name, c in outs:
        got = np.load(tmp_path / "all" / f"{name}.npy")
        assert got.dtype == np.float32 and np.array_equal(got, c.float().numpy())
    limit = 10 * (40 + 24) * 4  # room for 10 rows of both outputs
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), outs, limit, "_rank1")
    q = np.load(tmp_path / "a" / "qkv_rank1.npy")
    o = np.load(tmp_path / "a" / "o_rank1.npy")
    assert q.shape == (10, 40) and o.shape == (10, 24)
    assert np.array_equal(q[:, 0], o[:, 0]) and np.all(np.diff(q[:, 0]) > 0)
    assert np.array_equal(q, np.load(tmp_path / "b" / "qkv_rank1.npy"))


def test_reference_arm_honours_steps_and_dumps_its_output(tmp_path):
    out = run_bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path))
    assert out["steps"] == 1
    got = torch.from_numpy(np.load(tmp_path / "o.npy"))
    # the arm's seeded o_proj problem, through the same oracle
    _, n, k, _ = bench.LAYER[1]
    want = orc.nvfp4_gemm_ref_torch(*bench.cpu_case(torch.Generator().manual_seed(0), 16, n, k))
    assert got.dtype == torch.float32 and got.shape == (16, n)
    torch.testing.assert_close(got, want.float(), rtol=8e-3, atol=1e-3)


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True])
def test_gpu_arm_dumps_the_last_timed_step(tmp_path, graph):
    """Two timed steps over two weight copies: the files must hold the second step's GEMMs.
    They agree with the kernel on the rebuilt inputs to an output ulp: the benchmark's launches
    are PDL-chained, which moves the stream-K k-range cuts (fp4_gemm.cu, tilt_cuts), so the
    fp32 sums round differently from a standalone launch.  And they agree with the oracle."""
    import petit_kernel as pk

    steps = 2
    out = run_bench("--steps", str(steps), "--warmup", "1", "--no-details", "--dump-outputs",
                    str(tmp_path), *(["--graph"] if graph else []))
    assert out["steps"] == steps
    layers, copies, gs, acts, _ = bench.make_inputs(pk, bench.LAYER, 16, torch.device("cuda", 0), 0)
    assert copies == 2  # so the first and the last step used different weights
    for nm, n, k, _, b, sp in layers[(steps - 1) % copies]:
        got = torch.from_numpy(np.load(tmp_path / f"{nm}.npy"))
        assert got.shape == (16, n), nm
        c = pk.mul_nvfp4_a16(acts[k], b, sp, gs, 16, n, k, -1).float().cpu()
        assert (got - c).abs().max().item() <= c.abs().max().item() * 2 ** -7, nm
        w = pk.ops.dequant_dense(b, sp, 1.0, torch.bfloat16, n, k, False, True).float()
        assert orc.max_rel_err(got, ((acts[k].float() @ w.t()) * gs).cpu()) <= 1e-2, nm
