#!/bin/bash
# Runs the UNMODIFIED reference scripts of the original ViT-2SPN checkout at $V2S_REFERENCE_DIR through the launcher:
# pretraining (ssp_vit2spn_tiny.py) then fine-tuning (octmnist_ft_vit2spn.py), which loads the pretrained
# backbone the first one saved (ref:ssp_vit2spn_tiny.py:246 -> ref:octmnist_ft_vit2spn.py:190).  Logs go to $1.
# medmnist / fvcore / matplotlib may be absent and there may be no network, hence synthetic data (announced in the
# logs) and random-init weights.
set -u
ROOT="$(cd "$(dirname "$0")/.." && pwd)"
OUT="${1:?usage: run_reference_scripts.sh LOG_DIR}"
REF="${V2S_REFERENCE_DIR:?set V2S_REFERENCE_DIR to a checkout of the original ViT-2SPN}"
mkdir -p "$OUT"
WORK="${V2S_WORKDIR:-$(mktemp -d)}"
mkdir -p "$WORK"
cd "$WORK"
export PYTHONPATH="$ROOT" V2S_SYNTHETIC_DATA=1 V2S_ALLOW_RANDOM_INIT=1
status=0
for spec in "ssp_vit2spn_tiny.py:${V2S_SSP_DATASET_SIZE:-256}" "octmnist_ft_vit2spn.py:${V2S_FT_DATASET_SIZE:-4000}"; do
  script="${spec%%:*}"; size="${spec##*:}"
  [ -f "$REF/$script" ] || { echo "missing $REF/$script" | tee "$OUT/${script%.py}.log"; status=1; continue; }
  t0=$(date +%s)
  V2S_SHIM_DATASET_SIZE=$size timeout "${V2S_SCRIPT_TIMEOUT:-900}" python -m vit2spn.run "$REF/$script" \
      > "$OUT/${script%.py}.log" 2> "$OUT/${script%.py}.err"
  rc=$?
  echo "== $script rc=$rc $(( $(date +%s) - t0 )) s (dataset cap $size)" | tee -a "$OUT/summary.txt"
  [ $rc -eq 0 ] || status=1
done
ls -la "$WORK/ssp_retinaloct_tbme/vit2spn_tiny/" >> "$OUT/summary.txt" 2>&1
exit $status
