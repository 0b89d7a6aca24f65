"""CPU: the checkpoint validator (motionmixerconv_b200/checkpoint.py) on state_dicts written by the REFERENCE modules (the golden
fixtures' parameters, tests/golden/make_golden.py); detects missing / reordered keys, wrong shapes, broken se2 aliases."""
import json

import numpy as np
import pytest
import torch

from motionmixerconv_b200 import checkpoint as CK
from tests.golden_util import Golden, golden_cases


@pytest.mark.parametrize("case", golden_cases())
def test_fixture_parameters_validate(case):
    g = Golden(case)
    sd = {k: torch.from_numpy(np.asarray(v)) for k, v in g.params.items()}
    assert CK.validate_state_dict(sd, g.family, g.cfg) == []


def test_reference_checkpoint_file_through_the_cli(tmp_path, capsys):
    for case in ("conv_k1", "conv_k3_bn"):      # harmonic encoder + se2 aliases; BatchNorm buffers + se2 aliases
        g = Golden(case)
        cfg = json.loads(json.dumps(g.cfg))
        sd = {k: torch.from_numpy(np.array(v)) for k, v in g.params.items()}
        path = tmp_path / (case + ".pt")
        torch.save(sd, path)
        assert CK.main([str(path), "--family", "conv", "--cfg", json.dumps(cfg)]) == 0
        assert "OK" in capsys.readouterr().out
        bad = dict(sd)
        bad["Mixer_Block.0.se2.excitationBlock.0.weight"] = sd["Mixer_Block.0.se2.excitationBlock.0.weight"] + 1.0      # alias broken
        bad["LN.weight"] = torch.zeros(7)                                                                                # wrong shape
        del bad["fc_out.bias"]                                                                                           # missing
        problems = CK.validate_state_dict(bad, "conv", cfg)
        text = "\n".join(problems)
        assert "missing keys" in text and "LN.weight: shape" in text and "se2" in text
        reordered = dict(reversed(list(sd.items())))
        assert any("key order" in p for p in CK.validate_state_dict(reordered, "conv", cfg))
