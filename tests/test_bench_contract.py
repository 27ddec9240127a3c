"""``bench.py``'s command-line contract.  Without a GPU: the reference arm really tries to import the reference
and reports the exception text; the documented flags exist; the flagship config is the model BASELINE.json
names.  On a GPU: ``--steps`` is the number of timed steps and ``--dump-outputs`` writes the last step's outputs."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def _run(*args):
    return subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, timeout=300)


def test_reference_arm_prints_one_json_line_with_the_real_reason():
    out = _run("--impl", "reference", "--gpus", "1", "--steps", "5", "--warmup", "3")
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["n_gpus"] == 1
    if "unavailable" in line:                     # this image: spaCy / thinc / Ray are not installable
        why = line["unavailable"]
        assert "baseline/_ref" in why
        assert "does not exist" in why or "ModuleNotFoundError" in why or "ImportError" in why or "could not be driven" in why
    else:                                         # an image with the wheels: a real measurement
        assert line["value"] > 0 and line["unit"]


def test_cli_surface_the_driver_uses():
    out = _run("--help")
    assert out.returncode == 0
    for flag in ("--gpus", "--steps", "--warmup", "--impl", "--config", "--no-own-baseline", "--dump-outputs"):
        assert flag in out.stdout, flag


def test_flagship_config_is_the_named_model():
    sys.path.insert(0, str(ROOT))
    import argparse

    import bench
    from spacy_ray_b200.config import Config

    ns = argparse.Namespace(docs_per_gpu=1024, width=256, depth=8, min_len=8, max_len=40, dropout=0.1)
    cfg = Config().from_str(bench.flagship_config(ns, 0), interpolate=False)
    assert cfg["nlp"]["pipeline"] == ["ner"] or "ner" in cfg["nlp"]["pipeline"]
    t2v = cfg["components"]["ner"]["model"]["tok2vec"]
    assert "MultiHashEmbed" in t2v["embed"]["@architectures"] and t2v["embed"]["width"] == 256
    assert "MaxoutWindowEncoder" in t2v["encode"]["@architectures"]
    assert t2v["encode"]["width"] == 256 and t2v["encode"]["depth"] == 8 and t2v["encode"]["maxout_pieces"] == 3
    base = json.loads((ROOT / "BASELINE.json").read_text())
    assert "tok2vec+NER" in base["metric"]


def test_zero_steps_is_rejected():
    out = _run("--steps", "0")
    assert out.returncode != 0 and "--steps" in out.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("impl", ["ours", "nccl-baseline"])
def test_steps_are_timed_and_last_step_outputs_dumped(tmp_path, impl):
    small = ("--docs-per-gpu", "64", "--no-e2e", "--no-own-baseline", "--baseline-steps", "2")
    dumps = []
    for run in ("a", "b"):
        out = _run("--impl", impl, "--gpus", "1", "--steps", "3", "--warmup", "3", *small,
                   "--dump-outputs", str(tmp_path / run))
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads(out.stdout.strip().splitlines()[-1])
        assert line["impl"] == impl and line["steps"] == 3       # --baseline-steps caps only the context arm
        dumps.append({f.name: np.load(f) for f in sorted((tmp_path / run).iterdir())})
    a, b = dumps
    assert set(a) == {"losses.npy", "params.npy"} and sum(x.nbytes for x in a.values()) <= 64 << 20
    assert a["losses.npy"].dtype == np.float32 and a["params.npy"].dtype == np.float32
    assert a["losses.npy"].shape == (1,) and np.isfinite(a["losses.npy"]).all() and a["losses.npy"][0] > 0
    assert a["params.npy"].shape == b["params.npy"].shape and np.isfinite(a["params.npy"]).all()
    # same arguments, same inputs: two runs agree up to the order of floating-point accumulation
    assert np.allclose(a["losses.npy"], b["losses.npy"], rtol=1e-2)
    assert np.abs(a["params.npy"] - b["params.npy"]).max() < 1e-2
