"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports every declared symbol, the product
package never touches oracle/, the host-side mirror keeps the reference's names / state_dict keys / errors."""
import ast
import ctypes
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols(headers=("etude_b200.h", "etude_b200_kernels.h")):
    names = []
    for hdr in headers:
        src = open(os.path.join(ROOT, "include", hdr)).read()
        src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
        names += re.findall(r"\b(etude_[a-z0-9_]+)\s*\(", src)
    return sorted(set(names))


def test_library_loads_and_exports_every_declared_symbol():
    import __graft_entry__ as g
    g.build()
    from etude_b200 import _lib
    lib = _lib.load()
    declared = _declared_symbols()
    assert len(declared) >= 12
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/*.h but not exported"
    assert sorted(_lib.SIGNATURES) == declared, "ctypes table and headers disagree"
    # the test-only build exports the same ABI plus include/etude_b200_dev.h; none of the latter is in the product
    dev = _lib.load_dev()
    dev_only = _declared_symbols(("etude_b200_dev.h",))
    assert sorted(_lib.DEV_SIGNATURES) == dev_only and len(dev_only) >= 4
    for name in declared + dev_only:
        assert hasattr(dev, name), f"{name} missing from libetude_b200_dev.so"
    for name in dev_only:
        assert not hasattr(lib, name), f"{name} (debug entry point) leaked into the product library"
    assert b"sm_100a" in lib.etude_version()
    assert lib.etude_feature_rows(3840000) == 15360 + 64 and lib.etude_feature_rows(480000) == 2048 + 64


def test_create_fails_loudly_without_a_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from etude_b200 import _lib
    lib = _lib.load()
    blob = np.zeros(5614878, np.float32)
    h = ctypes.c_void_p()
    assert lib.etude_create(0, blob.ctypes.data, blob.size, ctypes.byref(h)) != 0
    assert len(lib.etude_last_error()) > 0
    from etude_b200 import AMTAPC_Extractor, ExtractorConfig
    with pytest.raises(RuntimeError):
        AMTAPC_Extractor(ExtractorConfig(), "/nonexistent.pth", device="auto")
    with pytest.raises(RuntimeError):
        AMTAPC_Extractor(ExtractorConfig(), "/nonexistent.pth", device="cpu")


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "etude_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            path = os.path.join(dirpath, f)
            if f.endswith(".py"):
                tree = ast.parse(open(path).read())
                for node in ast.walk(tree):
                    mods = []
                    if isinstance(node, ast.Import):
                        mods = [a.name for a in node.names]
                    elif isinstance(node, ast.ImportFrom):
                        mods = [node.module or ""]
                    assert not any(m.split(".")[0] == "oracle" for m in mods), f"{path} imports oracle"
            elif f.endswith((".cu", ".cuh", ".h")):
                assert "oracle" not in open(path).read(), f"{path} mentions oracle"


def test_state_dict_keys_and_checkpoint_roundtrip(tmp_path):
    from etude_b200.model import Decoder_SPEC2MIDI, Encoder_SPEC2MIDI, _Spec2MIDI
    from etude_b200.weights import STATE_DICT_LAYOUT, pack_state_dict
    from oracle import model as omodel
    model = _Spec2MIDI(Encoder_SPEC2MIDI(), Decoder_SPEC2MIDI())
    assert list(model.state_dict().keys()) == [k for k, _ in STATE_DICT_LAYOUT]
    sd = omodel.init_state_dict(3)
    p = tmp_path / "ckpt.pth"
    torch.save(sd, p)
    model.load_state_dict(torch.load(p, weights_only=True), strict=False)
    blob, missing = pack_state_dict(model._flat_state_dict(), strict=True)
    assert not missing and blob.shape == (5614878,)
    off = 0
    for k, shape in STATE_DICT_LAYOUT:
        n = int(np.prod(shape))
        assert np.array_equal(blob[off : off + n], sd[k].numpy().reshape(-1)), k
        off += n
    # partial checkpoints keep defaults (reference: strict=False); bad shapes raise
    blob2, missing2 = pack_state_dict({"encoder.conv.bias": torch.ones(4)})
    assert len(missing2) == len(STATE_DICT_LAYOUT) - 1 and np.all(blob2[20:24] == 1)
    with pytest.raises(ValueError):
        pack_state_dict({"encoder.conv.bias": torch.ones(5)})


def test_config_mirror_matches_reference_defaults_and_rejects_other_shapes():
    from etude_b200 import config as cfg
    c = cfg.ExtractorConfig()
    assert (c.feature.sr, c.feature.hop_sample, c.feature.fft_bins, c.feature.mel_bins) == (16000, 256, 2048, 256)
    assert (c.input.margin_b, c.input.margin_f, c.input.num_frame, c.input.min_value) == (32, 32, 512, -18.0)
    assert (c.infer.onset_threshold, c.infer.offset_threshold, c.infer.frame_threshold, c.infer.min_duration) == (0.5, 1.0, 0.5, 0.08)
    cfg.validate(c)
    c.input.num_frame = 128
    with pytest.raises(ValueError):
        cfg.validate(c)
    from etude_b200.model import Encoder_SPEC2MIDI
    with pytest.raises(ValueError):
        Encoder_SPEC2MIDI(hid_dim=128)


def test_reference_config_object_is_accepted():
    """The reference's `load_config().extractor` is a pydantic tree, not our dataclasses: validate() must accept any
    object with the same attributes.  tests/golden/reference_extractor_config.json holds the values of that object
    (etude/config/schema.py:68-131, SURVEY.md section 8), the ones the reference ran with when it made the other goldens;
    it is read back as a plain attribute tree, and the mirror's defaults must equal it field for field."""
    import json
    from types import SimpleNamespace

    from etude_b200 import config as cfg
    with open(os.path.join(ROOT, "tests", "golden", "reference_extractor_config.json")) as f:
        ref = json.load(f, object_hook=lambda d: SimpleNamespace(**d))
    assert cfg.validate(ref) is ref
    mine = cfg.ExtractorConfig()
    for section, fields in vars(ref).items():
        for name, value in vars(fields).items():
            assert getattr(getattr(mine, section), name) == value, f"extractor.{section}.{name}"


def test_window_bookkeeping_matches_reference_padding():
    from etude_b200.engine import feature_rows
    for n, t_pad in [(480000, 2048), (3840000, 15360), (1025, 512), (256 * 511, 512), (256 * 512, 1024)]:
        assert feature_rows(n) == t_pad + 64
        t = 1 + n // 256
        assert len(range(0, t, 512)) == t_pad // 512
