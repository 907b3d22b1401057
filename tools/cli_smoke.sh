#!/bin/bash
# End-to-end smoke of the drop-in CLI on a GPU box: generate-config -> synthetic .npy pool -> `dquartic train` (2 epochs,
# checkpoints in the reference format) -> resume from the latest checkpoint -> train with the weight EMA -> `dquartic predict`.
# Shrunken m/z axis (640) so checkpoints stay small.
set -e
ROOT=$(cd "$(dirname "$0")/.." && pwd)
export PYTHONPATH=$ROOT/diffusion-deconvolution-dia-msms-data_b200:$PYTHONPATH
W=${1:-/tmp/dq_cli_smoke}
rm -rf $W && mkdir -p $W && cd $W
python -m dquartic.cli generate-config cfg.json
python - <<'PY'
import json, numpy as np, sys
sys.path.insert(0, ".")
from dquartic.utils.synthetic import synth_pool
ms2, ms1 = synth_pool(24, 34, 640, seed=7, density=0.2)
np.save("ms2.npy", ms2); np.save("ms1.npy", ms1)
c = json.load(open("cfg.json"))
c["model"]["UNet1d"]["downsample_dim"] = 640
c["model"].update(batch_size=8, num_epochs=2, warmup_epochs=1, checkpoint_path="ckpt/best_model.ckpt")
c["wandb"]["use_wandb"] = False
c["data"]["parquet_directory"] = None   # the generated default points at a parquet directory; NPY paths are exclusive with it
json.dump(c, open("cfg.json", "w"), indent=1)
PY
mkdir -p ckpt
python -m dquartic.cli train --ms2-data-path ms2.npy --ms1-data-path ms1.npy cfg.json 2>&1 | tail -12
ls -la ckpt
python -m dquartic.cli train --ms2-data-path ms2.npy --ms1-data-path ms1.npy --batch-size 4 cfg.json 2>&1 | tail -6
python - <<'PY'
import torch
ck = torch.load("ckpt/dquartic_latest_checkpoint.ckpt", map_location="cpu", weights_only=False)
print("checkpoint keys", sorted(ck.keys()), "epoch", ck["epoch"], "n state entries", len(ck["model_state_dict"]))
assert len(ck["model_state_dict"]) == 396
PY
# train with the weight EMA, then deconvolve the pool with it (--weights auto picks the EMA)
mkdir -p ckpt_ema
python -m dquartic.cli train --ms2-data-path ms2.npy --ms1-data-path ms1.npy --checkpoint-path ckpt_ema/best_model.ckpt \
    --ema-decay 0.99 cfg.json 2>&1 | tail -3
python -m dquartic.cli predict --checkpoint-path ckpt_ema/best_model.ckpt --ms2-data-path ms2.npy --ms1-data-path ms1.npy \
    --output pred.npy --num-steps 10 --chunk 4 cfg.json
python - <<'PY'
import numpy as np
p, ms2 = np.load("pred.npy"), np.load("ms2.npy")
print("predicted", p.shape, p.dtype, "range", float(p.min()), float(p.max()))
assert p.shape == ms2.shape and p.dtype == np.float32 and np.isfinite(p).all()
PY
# hold out 25 % of the pool (6 slices: 15 pairs), select the best checkpoint by the EMA's validation loss, then score it
mkdir -p ckpt_val
python - <<'PY'
import json
c = json.load(open("cfg.json"))
c["validation"] = {"fraction": 0.25, "windows": 12, "bands": 5, "seed": 3}
json.dump(c, open("cfg_val.json", "w"), indent=1)
PY
python -m dquartic.cli train --ms2-data-path ms2.npy --ms1-data-path ms1.npy --checkpoint-path ckpt_val/best_model.ckpt \
    --ema-decay 0.99 cfg_val.json 2>&1 | grep -E "Validation|Best model"
python -m dquartic.cli evaluate --checkpoint-path ckpt_val/best_model.ckpt --ms2-data-path ms2.npy --ms1-data-path ms1.npy \
    --weights both --num-steps 10 --chunk 4 --output eval.json cfg_val.json
python - <<'PY'
import json, math, torch
r = json.load(open("eval.json"))
ck = torch.load("ckpt_val/best_model.ckpt", map_location="cpu", weights_only=False)
print("evaluate:", {w: (v["val_loss"], v["samplers"]["dpm++2m@10"]["mean"]) for w, v in r["results"].items()})
assert r["windows"] == 12 and r["results"]["ema"]["val_loss"] == ck["val_loss"] == ck["best_loss"]
assert all(math.isfinite(x) for v in r["results"].values() for l in v["samplers"]["dpm++2m@10"]["per_window"].values()
           for x in l)
PY
echo CLI_SMOKE_OK
