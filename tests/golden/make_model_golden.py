"""Generates tests/golden/model_golden.pt by running the REFERENCE'S OWN cubercnn modeling code
(/root/reference, unmodified) on oracle/d2lite (see oracle/ref_runner.py) on seeded synthetic inputs.

Pins oracle/cubercnn_oracle (tests/test_model_oracle.py) and, through it, the CUDA path.
Run here only:   python tests/golden/make_model_golden.py
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import model_io, ref_runner  # noqa: E402
from omni3d_b200 import synth  # noqa: E402

CASES = {"dla34": ("configs/cubercnn_DLA34_FPN.yaml", (128, 160)), "resnet34": ("configs/cubercnn_ResNet34_FPN.yaml", (128, 128))}


def main():
    torch.set_num_threads(8)        # = FIXTURE_THREADS of tests/test_model_oracle.py (results depend on the thread count)
    out = {}
    for name, (cfg_file, (H, W)) in CASES.items():
        cfg = ref_runner.reference_cfg(cfg_file)
        torch.manual_seed(0)
        model = ref_runner.build_reference_model(cfg)
        from detectron2.utils.events import EventStorage
        sd = model.state_dict()
        rec = {"init_sum": {k: float(v.double().sum()) for k, v in sd.items()},
               "init_abs": {k: float(v.double().abs().sum()) for k, v in sd.items()},
               "n_params": sum(p.numel() for p in model.parameters())}
        model.train()
        items = synth.make_batch(2, H, W, num_gt=4, seed=1)
        torch.manual_seed(123)
        with EventStorage(0) as st:
            losses = model(model_io.to_d2_inputs(items))
            sum(losses.values()).backward()
            rec["scalars"] = st.latest()
        rec["losses"] = {k: v.detach().clone() for k, v in losses.items()}
        rec["grad_norm"] = {n: float(p.grad.double().norm()) for n, p in model.named_parameters() if p.grad is not None}
        rec["no_grad"] = sorted(n for n, p in model.named_parameters() if p.grad is None)
        model.eval()
        with torch.no_grad():
            res = model(model_io.to_d2_inputs(synth.make_batch(2, H, W, with_gt=False, seed=3)))
        rec["detections"] = [{k: (v.tensor if hasattr(v, "tensor") else v).clone()
                              for k, v in r["instances"].get_fields().items()} for r in res]
        out[name] = rec
        print(name, rec["n_params"], {k: round(float(v), 6) for k, v in rec["losses"].items()},
              [len(d["scores"]) for d in rec["detections"]])
    torch.save(out, os.path.join(ROOT, "tests/golden/model_golden.pt"))
    print("wrote tests/golden/model_golden.pt")


if __name__ == "__main__":
    main()
