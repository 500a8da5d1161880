"""Drop-in proof against the REFERENCE'S OWN classes (SURVEY.md §8b).

tests/golden/dropin_reference.json records what the reference framework did with the plugin classes
(oracle/gen_golden_dropin.py, run with the unmodified reference: elliot's own BaseRecommenderModel, RecMixin, DataSet,
ModelCoordinator and run_experiment, with `external_models_path` pointing at elliot_b200/external/__init__.py).
The same case runs here on the stand-alone mirror, in a fresh interpreter with CUDA hidden, and has to agree:

  * the plugin classes implement every abstract method of elliot's BaseRecommenderModel ABC;
  * the kernel-side data views (`train_csr_of`, `eval_csr_of`) and the id order equal what elliot's own DataSet gave
    for the same frames, both from the mirror DataSet and from an object carrying only the attributes elliot's DataSet
    has (the models must not rely on mirror-only helpers);
  * a YAML whose model key is `external.BPRMF` gets through the run_experiment pipeline, plugin discovery included,
    and fails only at the CUDA check ("needs a CUDA device": there is no CPU fallback), as it did under
    elliot's ModelCoordinator and run_experiment;
  * past the availability check the constructor runs the host-side init and dies only in device code;
  * `autoset_params()` fills the attributes as elliot's did, and `name` follows the reference's own shortcut format
    (the reference BPRMF class's `name` evaluated on the same attributes).
"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "dropin_reference.json")

SCRIPT = r'''
import json, sys
sys.path.insert(0, sys.argv[1])
from oracle.gen_golden_dropin import plugin_facts
print("RESULT " + json.dumps(plugin_facts()))
'''


def test_plugin_classes_are_driven_by_the_reference_framework():
    with open(GOLDEN) as fh:
        ref = json.load(fh)
    r = subprocess.run([sys.executable, "-c", SCRIPT, ROOT], capture_output=True, text=True, timeout=600,
                       env={**os.environ, "CUDA_VISIBLE_DEVICES": ""})
    line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")]
    assert line, r.stdout[-2000:] + r.stderr[-3000:]
    out = json.loads(line[-1][7:])
    assert out["host"] == "standalone"
    assert out["abstract_methods"] == ref["abstract_methods"]
    assert set(out["classes"]) >= {"BPRMF", "BPRMF_batch", "MF2020", "MultiVAE", "NeuMF"}
    assert set(out["classes"]) == set(ref["classes"])
    for name, c in out["classes"].items():
        assert c["subclass"] and c["mixin"] and c["abstract_left"] == [], (name, c)
        assert ref["classes"][name] == c, (name, ref["classes"][name])
    assert ref["dataset_has_helper_methods"] is False
    for views in (out, out["plain"]):
        for k in ("train_csr", "eval_csr", "users", "items"):
            assert views[k] == ref[k], k
    for k in ("model_coordinator", "run_experiment"):
        assert "needs a CUDA device" in ref[k], ref[k]
    assert "needs a CUDA device" in out["construct"], out["construct"]
    assert out["run_experiment"] == ref["run_experiment"], out["run_experiment"]
    for facts in (ref, out):
        assert facts["ctor_after_check"] != "ran" and "AttributeError" not in facts["ctor_after_check"], facts["ctor_after_check"]
    assert out["autoset"] == ref["autoset"] == {"factors": 8, "lr": 0.05, "u_reg": 0.0025}
    assert out["name"] == ref["name"], (out["name"], ref["name"])
