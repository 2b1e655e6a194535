"""Argument checks of the seeded device decode loop (generate.py): rejected on the host before any model or device work."""
import pytest
import torch

from tcavp_b200 import generate as G


@pytest.mark.parametrize("kw,msg", [(dict(seed=1, kv_cache=False), "kv_cache"),
                                    (dict(seed=1, generator=torch.Generator()), "generator"),
                                    (dict(seed=1.5), "int"),
                                    (dict(seed=True), "int")])
def test_seed_argument_combinations_raise_before_any_launch(kw, msg):
    # model=None: the checks must fire before the engine is touched
    with pytest.raises(ValueError, match=msg):
        G.generate_ids(None, torch.zeros(1, 4, 8), torch.zeros(1, 3, dtype=torch.long), max_new_tokens=4, **kw)
