"""Acceptance: the reference's own inference scripts run UNCHANGED on top of the drop-in `src.*` package.

`src/inference/gen_george.py` and `src/inference/vis_george_sink.py` are executed with runpy exactly as shipped
(`__graft_entry__.build()` stages unmodified copies from a reference checkout into the git-ignored oracle/_ref/,
oracle/stage_reference.py; the scripts are never committed, so the tests skip where none were staged).  Everything they
touch is resolved as in a real checkout: hydra `_target_` paths -> the drop-in modules, `transformers.LlamaTokenizer`
from a tokenizer directory, HF / diffusers / torch checkpoints from `pretrained/…`, `data/json/val.jsonl`, and they
write `output/val_0/NN.jpg`.  Widths are reduced (tests/acceptance_fixture.py); resolutions, token counts, the
25-turn story length, the 8-image window, 50 Euler steps and (sink script) the KV slicing are the scripts' own."""
import importlib.util
import os
import re
import subprocess
import sys

import pytest

from oracle.stage_reference import STAGED as SCRIPTS

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "seed-story_b200")


@pytest.fixture(scope="module")
def project(tmp_path_factory, cuda_dev):
    root = str(tmp_path_factory.mktemp("seedstory_project"))
    for p in (os.path.join(PKG, "shims"), PKG, os.path.dirname(__file__)):
        if p not in sys.path:
            sys.path.insert(0, p)
    import acceptance_fixture
    info = acceptance_fixture.build_project(root, n_stories=1, n_captions=27)
    stubs = os.path.join(root, "_stubs")
    if importlib.util.find_spec("matplotlib") is None:      # imported (never used) by vis_george_sink.py:10
        os.makedirs(os.path.join(stubs, "matplotlib"), exist_ok=True)
        open(os.path.join(stubs, "matplotlib", "__init__.py"), "w").close()
        open(os.path.join(stubs, "matplotlib", "pyplot.py"), "w").close()
    return root, stubs, info


def _run_script(name, project):
    root, stubs, _ = project
    script = os.path.join(SCRIPTS, name)
    if not os.path.exists(script):
        pytest.skip(f"{script} not staged (__graft_entry__.build() stages it where a reference checkout is readable)")
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(PKG, "shims"), PKG, stubs, env.get("PYTHONPATH", "")])
    env["SEEDSTORY_PROJECT_ROOT"] = PKG          # pyrootutils.setup_root(): the reference tree has no .project-root
    env.pop("SEEDSTORY_SYNTHETIC", None)         # every checkpoint path must resolve to a real file
    code = f"import runpy; runpy.run_path({script!r}, run_name='__main__')"
    r = subprocess.run([sys.executable, "-c", code], cwd=root, env=env, capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, f"{name} failed:\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}"
    return r


def test_gen_george_runs_unchanged(project):
    r = _run_script("gen_george.py", project)
    out = os.path.join(project[0], "output", "val_0")
    imgs = sorted(f for f in os.listdir(out) if re.fullmatch(r"\d\d\.jpg", f))
    # story_len 25: the loop runs until 24 images exist (gen_george.py:205-229) because every turn emits an image
    assert imgs[0] == "01.jpg" and len(imgs) == 24, imgs
    from PIL import Image
    im = Image.open(os.path.join(out, "ori_01.jpg"))
    assert im.size == (1024, 1024)
    lines = open(os.path.join(out, "token.txt")).read().strip().splitlines()
    assert len(lines) == 24 and lines[0].startswith("context token: torch.Size([1, ")
    # window of 8 images: the prompt grows turn by turn (text + 66 image tokens) until the oldest image is evicted
    # every turn (gen_george.py:233-237), from where on its length stays put
    ctx = [int(l.split(",")[1].strip(" ])")) for l in lines]
    assert ctx[1] > ctx[0] + 66 and ctx[7] > ctx[1], ctx
    assert max(ctx[10:]) - min(ctx[10:]) <= 32 and max(ctx) <= ctx[0] + 9 * (66 + 120), ctx
    assert "Init adapter pipe done" in r.stdout


def test_vis_george_sink_runs_unchanged(project):
    r = _run_script("vis_george_sink.py", project)
    out = os.path.join(project[0], "output", "val_0")
    lines = open(os.path.join(out, "token.txt")).read().strip().splitlines()
    assert any("boi_idx" in l for l in lines), "vis_george_sink.py writes boi_idx into token.txt (:236)"
    n_sink = sum("boi_idx" in l for l in lines)
    assert n_sink == 23, (n_sink, lines[-3:])     # first generate + 22 loop turns (break at text_id >= 24, :253)
    assert os.path.exists(os.path.join(out, "23.jpg"))
