#!/bin/bash
# Config 4 before and after a change to the sequence-first finish: the parent commit against this tree, in one GPU
# session.
#
#   tools/c4_finish_ab.sh export [REV]   # with git: export REV (default HEAD) into ab_parent/ (git-ignored)
#   tools/c4_finish_ab.sh run [OUT]      # on the GPU: build both trees, then measure; results under OUT
#                                        # (default ab_out/, git-ignored)
#
# run: three alternated pairs of `bench.py --no-others --no-cpu-baseline --no-e2e --no-api` (parent, then this tree),
# one `tools/c4_order_ab.py --trace` per tree for the kernel breakdown, one short `--dump-outputs` run per tree to
# compare the hits byte for byte, then one plain `bench.py` of this tree for the record.  summary.json holds the card
# name and power limit, ms per step per run, medians and spreads, the threshold sweeps and the finish kernel's time.
set -eu
REPO=$(cd "$(dirname "$0")/.." && pwd)
PARENT=$REPO/ab_parent
cd "$REPO"

case "${1:-}" in
export)
    rm -rf "$PARENT"
    mkdir -p "$PARENT"
    git archive "${2:-HEAD}" | tar -x -C "$PARENT"
    echo "exported $(git rev-parse --short "${2:-HEAD}") into ab_parent/"
    exit 0 ;;
run) ;;
*) echo "usage: $0 export [REV] | run [OUT]" >&2; exit 2 ;;
esac

OUT=$(mkdir -p "${2:-ab_out}" && cd "${2:-ab_out}" && pwd)
[ -d "$PARENT" ] || { echo "no ab_parent/: run '$0 export' first" >&2; exit 2; }
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > "$OUT/card.txt"
(cd "$PARENT" && python -c "import __graft_entry__ as g; g.build()")
python -c "import __graft_entry__ as g; g.build()"

AB="--no-others --no-cpu-baseline --no-e2e --no-api"
for i in 1 2 3; do
    (cd "$PARENT" && python bench.py $AB > "$OUT/parent_$i.json" 2> "$OUT/parent_$i.err")
    python bench.py $AB > "$OUT/branch_$i.json" 2> "$OUT/branch_$i.err"
done
(cd "$PARENT" && python tools/c4_order_ab.py --trace "$OUT/parent_kernels.json" > "$OUT/parent_order_ab.json")
python tools/c4_order_ab.py --trace "$OUT/branch_kernels.json" > "$OUT/branch_order_ab.json"
DUMP="--steps 2 --warmup 1 --no-others --no-cpu-baseline --no-e2e --no-api --no-sweep"
(cd "$PARENT" && python bench.py $DUMP --dump-outputs "$OUT/dump_parent" > /dev/null 2>&1)
python bench.py $DUMP --dump-outputs "$OUT/dump_branch" > /dev/null 2>&1
python bench.py > "$OUT/bench_default.json" 2> "$OUT/bench_default.err"

python - "$OUT" <<'PY'
import filecmp, json, os, sys
import numpy as np
out = sys.argv[1]
load = lambda name: json.load(open(os.path.join(out, name)))
runs = {t: [load("%s_%d.json" % (t, i)) for i in (1, 2, 3)] for t in ("parent", "branch")}
ms = {t: [r["ms_per_step"] for r in v] for t, v in runs.items()}
res = {"card": open(os.path.join(out, "card.txt")).read().strip(),
       "ms_per_step": {t: {"runs": v, "median": float(np.median(v)),
                           "spread": float((max(v) - min(v)) / np.median(v))} for t, v in ms.items()},
       "hits_rank0": {t: [r["hits_rank0"] for r in v] for t, v in runs.items()},
       "sweep": {t: v[-1].get("threshold_sweep_rank0") for t, v in runs.items()}}
res["branch_over_parent"] = res["ms_per_step"]["branch"]["median"] / res["ms_per_step"]["parent"]["median"]
res["every_branch_run_faster"] = max(ms["branch"]) < min(ms["parent"])
fin = {}
for t in ("parent", "branch"):
    k = load("%s_kernels.json" % t)["kernels"]["sequence_first"]
    fin[t] = {name: us for name, us in k.items() if "kmer_finish_kernel" in name}
res["finish_kernel_us"] = fin
names = sorted(os.listdir(os.path.join(out, "dump_parent")))
res["dump_files"] = names
res["dumps_identical"] = names == sorted(os.listdir(os.path.join(out, "dump_branch"))) and all(
    filecmp.cmp(os.path.join(out, "dump_parent", f), os.path.join(out, "dump_branch", f), shallow=False) for f in names)
with open(os.path.join(out, "summary.json"), "w") as fh:
    json.dump(res, fh, indent=1)
print(json.dumps(res, indent=1))
PY
