"""CPU tier: the C ABI must answer malformed input with an error code, never with a crash or a hang.  Valid compiled scenes
(the random scene graphs of tests/test_gpu_fuzz.py) are corrupted field by field — node types, child ranges and indices
(including cycles), material / texture / table ids, parameters set to NaN / inf / huge / negative, truncated arrays — and
pushed through rtb_scene_set_* + rtb_scene_build_bvh in a host-only scene.  Run in a subprocess so that a crash is a
test failure, not the end of the test session."""
import os
import subprocess
import sys
import textwrap

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))  # the child script imports from here and from tests/
SCRIPT = textwrap.dedent(r'''
    import sys, copy
    import numpy as np
    sys.path.insert(0, "tests")
    import ray_tracer_archive_b200 as rtb
    from ray_tracer_archive_b200 import scenes, scene as S, _ffi as F
    from test_gpu_fuzz import _random_scene

    first, last = int(sys.argv[1]), int(sys.argv[2])
    ctx = rtb.Context(0) if len(sys.argv) > 3 and sys.argv[3] == "gpu" else None
    outcomes = {"ok": 0, "error": 0}
    for seed in range(first, last):
        rng = np.random.default_rng(50000 + seed)
        world, lights = _random_scene(seed % 40, S, scenes, False, True, None)
        cs = rtb.compile_scene(world, lights)
        for trial in range(12):
            c = copy.copy(cs)
            c.nodes, c.child_index = cs.nodes.copy(), cs.child_index.copy()
            c.materials, c.textures, c.lights = cs.materials.copy(), cs.textures.copy(), cs.lights.copy()
            for _ in range(int(rng.integers(1, 4))):
                kind = int(rng.integers(0, 9))
                n = len(c.nodes)
                i = int(rng.integers(0, n))
                weird = [np.nan, np.inf, -np.inf, 1e308, -1e308, 0.0, -1.0, 1e-320][int(rng.integers(0, 8))]
                if kind == 0:
                    c.nodes["type"][i] = int(rng.integers(0, 70))
                elif kind == 1:
                    c.nodes["first_child"][i] = int(rng.integers(0, 2 ** 32, dtype=np.uint64))
                elif kind == 2:
                    c.nodes["n_children"][i] = int(rng.integers(0, 2 ** 32, dtype=np.uint64))
                elif kind == 3 and len(c.child_index):
                    c.child_index[int(rng.integers(0, len(c.child_index)))] = int(rng.integers(0, n + 3))  # may close a cycle
                elif kind == 4:
                    c.nodes["material"][i] = int(rng.integers(0, 2 ** 32, dtype=np.uint64))
                elif kind == 5:
                    c.nodes["p"][i][int(rng.integers(0, c.nodes["p"].shape[1]))] = weird
                elif kind == 6 and len(c.textures):
                    j = int(rng.integers(0, len(c.textures)))
                    f = ["type", "even", "odd", "table"][int(rng.integers(0, 4))]
                    c.textures[f][j] = int(rng.integers(0, 2 ** 32, dtype=np.uint64))
                elif kind == 7 and len(c.materials):
                    j = int(rng.integers(0, len(c.materials)))
                    f = c.materials.dtype.names[int(rng.integers(0, len(c.materials.dtype.names)))]
                    if c.materials[f].dtype.kind in "ui":
                        c.materials[f][j] = int(rng.integers(0, 2 ** 32, dtype=np.uint64))
                    else:
                        c.materials[f][j] = weird
                elif kind == 8:
                    c.root = int(rng.integers(0, n + 5))
            try:
                s = rtb.Scene(ctx, c)
                s.info()
                if ctx is not None:  # GPU tier: what the host accepted also renders (or is refused) without a hang
                    cam = rtb.Camera.new((2.0, 7.0, 19.0), (0.0, 2.0, 0.0), (0, 1, 0), 40.0, 1.5, 0.0, 19.0, 0.0, 1.0)
                    acc, st = s.render(cam, rtb.make_params(32, 24, 4, 12, (0.5, 0.6, 0.8), seed=seed))
                    assert st["paths"] == 32 * 24 * 4
                s.close()
                outcomes["ok"] += 1
            except rtb.RtbError:
                outcomes["error"] += 1
    print("outcomes", outcomes)
''')


@pytest.mark.parametrize("chunk", [0, 1, 2])
def test_corrupted_scene_records_never_crash(chunk):
    r = subprocess.run([sys.executable, "-c", SCRIPT, str(20 * chunk), str(20 * chunk + 20)], capture_output=True, text=True, timeout=900,
                       cwd=ROOT)
    assert r.returncode == 0, f"exit code {r.returncode}\n{r.stdout[-2000:]}\n{r.stderr[-3000:]}"
    assert "outcomes" in r.stdout
    print(r.stdout.strip().splitlines()[-1])


@pytest.mark.gpu
def test_corrupted_scenes_render_or_are_refused():
    """GPU tier: every corrupted scene the host accepts (parameters that are finite but absurd, odd but legal wiring) is
    rendered at 32x24x4 — the device must finish and account for every path."""
    r = subprocess.run([sys.executable, "-c", SCRIPT, "0", "40", "gpu"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, f"exit code {r.returncode}\n{r.stdout[-2000:]}\n{r.stderr[-3000:]}"
    print(r.stdout.strip().splitlines()[-1])
