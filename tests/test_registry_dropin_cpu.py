"""CPU: the plugin-level drop-in of INTEGRATION.md section 1, executed VERBATIM against the UNMODIFIED reference registries
(/root/reference/liteasr/models/__init__.py:53-86, criterions/__init__.py:28-56) loaded through ``oracle/ref_shims.py``.

Runs in a fresh interpreter (import order matters: ``liteasr_b200.config`` derives its dataclasses from
``liteasr.config.LiteasrDataclass`` when LiteASR is importable at that moment).  Skipped where no copy of the upstream LiteASR
source tree is found (``oracle/ref_shims.py``: ``LITEASR_REFERENCE_ROOT``).

The state_dict half of that check also runs without the upstream tree, against what the unmodified reference model recorded
when the golden files were generated (``oracle/make_golden.py``): its parameter names in ``named_parameters()`` order with
their shapes (``f64.grads``) and its BatchNorm buffers (``f64.bn``, ``f64.nbt``), for three model sizes."""
import json
import os
import subprocess
import sys
import textwrap

import pytest

from oracle import ref_shims

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SCRIPT = r'''
import dataclasses, re, sys, types
sys.path.insert(0, ROOT)
from oracle import ref_shims
ref_shims.install()

# a minimal working OmegaConf.merge for the stubbed omegaconf (hydra / omegaconf are not installed here): dataclass defaults
# overridden by the attributes of a duck-typed cfg; the result keeps `_parent` / `_content` in __dict__ like a DictConfig,
# because models/__init__.py:60-67 reads and writes exactly those two entries.
class Cfg:
    def __init__(self, **kw):
        self.__dict__["_parent"] = None
        self.__dict__["_content"] = {}
        for k, v in kw.items():
            setattr(self, k, v)
    def __setattr__(self, k, v):
        self.__dict__[k] = v
        self.__dict__["_content"][k] = v

class OmegaConf:
    @staticmethod
    def merge(dc, cfg):
        node = dc() if isinstance(dc, type) else dc
        out = Cfg(**{f.name: getattr(node, f.name) for f in dataclasses.fields(node)})
        for k, v in cfg.__dict__["_content"].items():
            setattr(out, k, v)
        return out
    @staticmethod
    def set_struct(cfg, flag):
        pass

sys.modules["omegaconf"].OmegaConf = OmegaConf
import liteasr.models as ref_models            # the unmodified reference registries (auto-import every reference model)
import liteasr.criterions as ref_criterions
assert "U2" in ref_models.MODEL_REGISTRY and ref_models.MODEL_REGISTRY["U2"].__module__ == "liteasr.models.u2"

# ---- INTEGRATION.md section 1, verbatim: the two python blocks become liteasr/models/u2_b200.py and
# ---- liteasr/criterions/hybrid_ctc_b200.py
text = open(ROOT + "/INTEGRATION.md").read()
sec = text.split("## 1.")[1].split("## 2.")[0]
blocks = re.findall(r"```python\n(.*?)```", sec, flags=re.S)
assert len(blocks) >= 2
for name, src in (("liteasr.models.u2_b200", blocks[0]), ("liteasr.criterions.hybrid_ctc_b200", blocks[1])):
    mod = types.ModuleType(name)
    sys.modules[name] = mod
    exec(compile(src, name, "exec"), mod.__dict__)

import liteasr_b200.models.u2 as b200_u2
import liteasr_b200.criterions.hybrid_ctc_attn as b200_crit
from liteasr.config import LiteasrDataclass
assert issubclass(b200_u2.U2Config, LiteasrDataclass) and issubclass(b200_crit.HybridCTCLossConfig, LiteasrDataclass)
from liteasr_b200.optims import AdamConfig, NoamConfig
assert issubclass(NoamConfig, AdamConfig) and issubclass(AdamConfig, LiteasrDataclass)
assert issubclass(ref_models.MODEL_REGISTRY["U2"], b200_u2.U2)
assert issubclass(ref_criterions.CRITERION_REGISTRY["hybrid_ctc"], b200_crit.HybridCTCLoss)
assert ref_models.MODEL_DATACLASS_REGISTRY["U2"] is b200_u2.U2Config

# ---- build through the REFERENCE's build_model / build_criterion with the values of config/model/my_U2.yaml
task = types.SimpleNamespace(feat_dim=80, vocab_size=4233)
mcfg = Cfg(name="U2", dropout_rate=DROPOUT, enc_arch="Conformer", use_rel=True, enc_dim=256, enc_ff_dim=2048, enc_attn_heads=4,
           enc_attn_dropout_rate=0.0, enc_layers=2, activation="swish", dec_arch="Transformer", dec_dim=256, dec_ff_dim=2048,
           dec_attn_heads=4, dec_self_attn_dropout_rate=0.0, dec_src_attn_dropout_rate=0.0, dec_layers=1)
model = ref_models.build_model(mcfg, task)
assert isinstance(model, b200_u2.U2) and type(model).__module__ == "liteasr.models.u2_b200"
assert model.sos == model.eos == 4232 and model.blank == 0 and model.ignore == -1
assert mcfg.__dict__["_content"]["input_dim"] == 80 and mcfg.__dict__["_content"]["vocab_size"] == 4233   # models/__init__.py:65-67
assert model.encoder.enc_layers[0].dropout_rate == DROPOUT and model.encoder.enc_layers[0].self_attn.dropout_rate == 0.0
assert model.encoder.enc_layers[0].feed_forward.dropout_rate == DROPOUT and model.ctc.dropout_rate == DROPOUT
assert model.decoder.dec_layers[0].dropout_rate == DROPOUT and model.decoder.dec_layers[0].src_attn.dropout_rate == 0.0
ccfg = Cfg(name="hybrid_ctc", smoothing=0.1, ctc_weight=0.3)
crit = ref_criterions.build_criterion(ccfg, task)
assert isinstance(crit, b200_crit.HybridCTCLoss) and crit.cfg.vocab_size == 4233 and crit.cfg.ctc_weight == 0.3
# state_dict schema = the reference model's own (same names and shapes)
ref_model_cls = sys.modules["liteasr.models.u2"].U2
rcfg = sys.modules["liteasr.models.u2"].U2Config(input_dim=80, vocab_size=4233, enc_layers=2, dec_layers=1)
for f in ref_shims._DROPOUT_FIELDS:
    setattr(rcfg, f, 0.0)
ref_sd = ref_model_cls(rcfg).state_dict()
sd = model.state_dict()
assert list(sd.keys()) == list(ref_sd.keys()), "state_dict keys/order differ from the reference model"
assert all(sd[k].shape == ref_sd[k].shape and sd[k].dtype == ref_sd[k].dtype for k in sd)
print("DROPIN-OK")
'''


@pytest.mark.skipif(not ref_shims.reference_available(), reason="needs the upstream LiteASR source tree (LITEASR_REFERENCE_ROOT)")
@pytest.mark.parametrize("dropout", [0.1])
def test_integration_md_section1_against_unmodified_reference_registry(dropout):
    src = f"ROOT = {ROOT!r}\nDROPOUT = {dropout!r}\n" + textwrap.dedent(SCRIPT)
    r = subprocess.run([sys.executable, "-c", src], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0 and "DROPIN-OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


@pytest.mark.parametrize("case", ["tiny", "tiny_odd", "c1"])
def test_state_dict_schema_matches_the_reference_recording(case):
    """Parameter names, order and shapes and the BatchNorm buffers of the product's U2 are the unmodified reference model's, as
    recorded in tests/golden/u2_<case>.json (enc / dec layers 2 / 2, 1 / 1 and 4 / 6).  The recording holds no dtypes and no
    position tables, so those two stay with the live check above."""
    from liteasr_b200.models.u2 import U2, U2Config
    with open(os.path.join(ROOT, "tests", "golden", f"u2_{case}.json")) as f:
        g = json.load(f)
    rec = g["f64"]
    model = U2(U2Config(**g["dims"]))
    assert [(k, list(p.shape)) for k, p in model.named_parameters()] == [(k, v["shape"]) for k, v in rec["grads"].items()]
    sd = model.state_dict()
    for group in (rec["bn"], rec["nbt"]):
        assert [k for k in sd if k in group] == list(group)
    assert all(list(sd[k].shape) == v["shape"] for k, v in rec["bn"].items())
    # the sinusoid position tables are the only entries the recording does not list
    recorded = set(rec["grads"]) | set(rec["bn"]) | set(rec["nbt"])
    assert all(k.endswith(".pe.pe") for k in sd if k not in recorded)
