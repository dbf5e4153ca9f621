"""Generates tests/golden/reference_schema.json by EXECUTING THE UNMODIFIED REFERENCE on CPU through oracle/refshim.py:
  * configs: configs/{two_head_model,quant_two_head_model,midi_conformer}.yaml flattened by the reference's own
    utils/config_utils.read_full_config, reduced to the keys synth.named_config defines (a key the reference lacks is
    left out, so the test sees it missing);
  * state_dict_shapes: name -> shape of modules/model/Gmidi_conform.midi_conforms built for the two_head config.
Outputs are committed; the reference is needed only to regenerate them.

    SOME_REFERENCE_ROOT=<reference checkout> python tests/golden/make_golden_schema.py
"""
import json
import os
import pathlib
import sys

HERE = pathlib.Path(__file__).resolve().parent
REPO = HERE.parent.parent
sys.path.insert(0, str(REPO))

from oracle import refshim  # noqa: E402
from some_b200 import synth  # noqa: E402

CONFIGS = {'two_head': 'two_head_model', 'quant_two_head': 'quant_two_head_model', 'midi_conformer': 'midi_conformer'}


def main():
    refshim.load_reference()
    from modules.model.Gmidi_conform import midi_conforms
    from utils.config_utils import read_full_config
    cwd = os.getcwd()
    os.chdir(refshim.REFERENCE_ROOT)                  # base_config entries are relative to the reference's root
    try:
        flat = {key: read_full_config(pathlib.Path(f'configs/{name}.yaml')) for key, name in CONFIGS.items()}
    finally:
        os.chdir(cwd)
    configs = {key: {k: flat[key][k] for k in synth.named_config(key) if k in flat[key]} for key in CONFIGS}
    cfg = synth.named_config('two_head')
    model = midi_conforms({'midi_extractor_args': dict(cfg['midi_extractor_args']), 'units_dim': 80, 'midi_num_bins': 128})
    shapes = {k: list(v.shape) for k, v in model.state_dict().items()}
    out = {'configs': configs, 'state_dict_shapes': shapes}
    (HERE / 'reference_schema.json').write_text(json.dumps(out, indent=1, sort_keys=True) + '\n')
    print({k: len(v) for k, v in configs.items()}, len(shapes), 'state_dict entries')


if __name__ == '__main__':
    main()
