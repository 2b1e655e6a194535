"""Host-side checks of FineTuner's gradient clipping / non-finite step skipping options: argument checks made before any device work,
and the workspace size the Python front end allocates against the one the C header declares.  Nothing here needs a GPU."""
import math
import os
import re

import pytest

import tcavp_b200 as T
from tcavp_b200 import ops

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("bad", [0, 0.0, -1.0, math.inf, -math.inf, math.nan])
def test_finetuner_rejects_max_grad_norm_that_is_not_finite_and_positive(bad):
    m = T.MultiModalTrajectoryModel(**T.MODEL_PRESETS["tiny"])       # stays on the CPU
    before = {n: p.data_ptr() for n, p in m.named_parameters()}
    with pytest.raises(ValueError, match="max_grad_norm"):
        T.FineTuner(m, max_grad_norm=bad, skip_nonfinite=True)
    # rejected before the parameters were moved into the flat buffer
    assert {n: p.data_ptr() for n, p in m.named_parameters()} == before


def test_clip_workspace_and_record_match_the_header():
    hdr = open(os.path.join(ROOT, "include", "tcavp.h")).read()
    assert int(re.search(r"#define\s+TCAVP_CLIP_WORKSPACE_BYTES\s+(\d+)", hdr).group(1)) == ops.CLIP_WORKSPACE_BYTES
    assert ops.CLIP_WORKSPACE_BYTES % 8 == 0
    rec = re.search(r"typedef struct \{(.*?)\} tcavp_clip_record;", hdr, re.S).group(1)
    fields = re.findall(r"^\s*(float|int)\s+(\w+);", rec, re.M)
    assert fields == [("float", "total_norm"), ("float", "clip_coef"), ("int", "skip"), ("int", "reserved")]
    assert ops.clip_record("cpu").shape == (4,)
