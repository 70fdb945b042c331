# ragged-batch timing on one GPU (scripts/varlen_time.py): bash scripts/gpu_varlen.sh [OUT_DIR] [STEPS]
# writes OUT_DIR/r03_varlen_time.json (the record profiles/ keeps) and OUT_DIR/varlen_time.log
cd "$(dirname "$0")/.."
OUT=${1:-$(mktemp -d)}  # (default: a fresh temporary directory, nothing is written into the tree)
mkdir -p "$OUT"
timeout 900 python scripts/varlen_time.py --steps "${2:-30}" --out "$OUT/r03_varlen_time.json" > "$OUT/varlen_time.log" 2>&1
echo "rc=$? record: $OUT/r03_varlen_time.json"; tail -3 "$OUT/varlen_time.log" | cut -c1-2000
