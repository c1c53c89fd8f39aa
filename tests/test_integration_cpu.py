"""CPU: the import seam of the drop-in modules.  `models/` is a PEP 420 namespace package both here and in the
original project, so with this repo's package directory ahead of a checkout on sys.path, `models.deep_sets` /
`models.graph_net` resolve to the B200 modules while the checkout's other modules (`models.wrapper`, `train`) still
resolve to the checkout.  A minimal stand-in checkout with that layout is written to a temporary directory."""
import os
import subprocess
import sys
import textwrap

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_models_namespace_resolves_to_b200_modules(tmp_path):
    ref = tmp_path / "checkout"
    (ref / "models").mkdir(parents=True)
    (ref / "models" / "wrapper.py").write_text("class ModelWrapper:\n    def __init__(self, model):\n        self.model = model\n")
    (ref / "train.py").write_text("from models.graph_net import GraphNet\nfrom models.deep_sets import DeepSets\n"
                                  "from models.wrapper import ModelWrapper\n")
    code = textwrap.dedent(f"""
        import sys
        sys.dont_write_bytecode = True
        sys.path[:0] = [{os.path.join(ROOT, 'point-cloud-classifier_b200')!r}, {str(ref)!r}]
        import train
        import models.deep_sets as ds, models.graph_net as gn, models.wrapper as mw
        assert "pcc_b200" in ds.DeepSets.__module__ and "pcc_b200" in gn.GraphNet.__module__
        assert mw.__file__.startswith({str(ref)!r}) and train.__file__.startswith({str(ref)!r})
        model = train.ModelWrapper(train.DeepSets(input_dim=6, phi_layers=[256, 256], rho_layers=[256], output_dim=1,
                                                  sparse_batching=True, pooling="mean", layer_norm=False,
                                                  activation="gelu", residual_block=True))
        assert type(model.model).__module__.startswith("pcc_b200")
        assert list(model.model.state_dict().keys())[:2] == ["phi.0.weight", "phi.0.bias"]
        g = train.GraphNet(input_dim=4, hidden_dim=128, output_dim=1, activation="tanh")
        assert type(g).__module__.startswith("pcc_b200")
        print("OK")
    """)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout + r.stderr
