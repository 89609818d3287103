"""tune_params --nms_thresh without a GPU: --help, the refusals of the threshold list before any frame is read, and the
output block of evaluate_settings with and without NMS thresholds."""
import itertools
import os
import subprocess
import sys

import numpy as np
import pytest

from findnpropagate_b200 import quality, synth, tune_params
from findnpropagate_b200.seeker import OutLayout

from test_extract_cli import HEAD
from test_tune_cpu import P, _grid, tools_dir  # noqa: F401  (tools_dir is a fixture)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_QUALITY = quality.QualitySpec(synth.CLASS_NAMES).n_counters
# the regions of the block before the NMS counters existed, in their order
REGIONS = ["boxes", "score", "best", "count", "npts", "nvalid", "status", "recall", "keep", "sel_boxes", "sel_score",
           "sel_best", "sel_count", "sel_recall", "sel_precision", "quality"]


def test_help_names_the_flag():
    r = subprocess.run([sys.executable, "-m", "findnpropagate_b200.tune_params", "--help"], cwd=ROOT,
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    assert "--nms_thresh" in r.stdout


@pytest.mark.parametrize("thresh,needle", [
    ([str(k / 10) for k in range(1, 10)], "at most 8"),
    (["0.1", "0.3", "0.1"], "0.1 is given twice"),
    (["0.1", "nan"], "nan"),
    (["inf"], "inf"),
])
def test_threshold_refusals_exit_1_before_any_frame_is_read(tools_dir, capsys, monkeypatch, thresh, needle):  # noqa: F811
    monkeypatch.setattr(tune_params, "build_feed", lambda *a, **k: pytest.fail("read frames"))
    monkeypatch.setattr(tune_params, "build_head", lambda *a, **k: pytest.fail("built the head"))
    with pytest.raises(SystemExit) as e:
        tune_params.main(["--cfg_file", HEAD, "--grid", _grid({P + "dns_w": [1.0]}), "--nms_thresh"] + thresh)
    assert e.value.code == 1
    err = capsys.readouterr().err
    assert needle in err and "--nms_thresh" in err


@pytest.mark.parametrize("F,S,n_quality", list(itertools.product((0, 1, 7, 300), (1, 3, 257), (0, N_QUALITY))))
def test_out_layout_without_thresholds_is_unchanged(F, S, n_quality):
    lay = OutLayout(F, 1, S, n_quality)
    assert list(lay.regions) == REGIONS
    assert OutLayout(F, 1, S, n_quality, 0).regions == lay.regions
    assert OutLayout(F, 1, S, n_quality, 0).nbytes == lay.nbytes
    # the NMS counters go after every existing region, which keep their offsets
    nms = OutLayout(F, 1, S, n_quality, 3)
    assert list(nms.regions) == REGIONS + ["nms_quality"]
    assert all(nms.regions[k] == lay.regions[k] for k in REGIONS)
    off, dt, shape = nms.regions["nms_quality"]
    assert off == lay.nbytes and dt == np.dtype(np.int64) and shape == (3, S, n_quality)
    assert nms.nbytes == lay.nbytes + 8 * 3 * S * n_quality
