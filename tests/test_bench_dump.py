"""bench.py --dump-outputs: the arrays of the last timed step, as .npy files two builds can be compared by."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")


def test_bad_arguments_are_refused_before_any_work():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        r = subprocess.run([sys.executable, BENCH, "--gpus", "1"] + extra, capture_output=True, text=True, timeout=300)
        assert r.returncode == 2, (extra, r.stderr[-2000:])


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step(tmp_path):
    from canonicalsg2im_b200 import synth
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, BENCH, "--gpus", "1", "--steps", "2", "--warmup", "3", "--configs", "none",
                        "--no-cpu-baseline", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2
    files = sorted(os.listdir(out))
    assert sum(os.path.getsize(out / f) for f in files) <= 64 << 20
    a = {f[:-len(".npy")]: np.load(out / f) for f in files}
    assert all(x.dtype in (np.float32, np.float64) and np.isfinite(x).all() for x in a.values())
    assert a["loss"].shape == () and a["loss"] > 0
    assert a["triples_after_canon"] == line["triples_after_canon_rank0"]
    # every parameter of the model and of the generator's embedding, moved off the seeded initial state by Adam
    init = synth.make_state(synth.Vocab(42), seed=0)
    init.update({"layout_embedding." + k: v for k, v in synth.make_layout_state(synth.Vocab(42), 128, seed=0).items()})
    for k in ("gconvs.0.net1.0.weight", "box_net.2.bias", "attribute_embedding.att_emb_0.weight",
              "layout_embedding.att_emb_0.weight"):
        name = "param." + (k if k.startswith("layout_embedding.") else "model." + k)
        got, ref = a[name], init[k]
        assert got.shape == ref.shape and not np.array_equal(got, ref), k
        assert np.abs(got - ref).max() < 0.05 * np.abs(ref).max(), k
