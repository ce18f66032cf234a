# Fine-tuning: build, the fine-tuning GPU tests, the rest of the GPU suite, tools/time_finetune.py, smoke() and one bench
# line.  Logs go to the directory given as the first argument (default: a fresh temporary directory).
set -u
out="${1:-$(mktemp -d)}"
mkdir -p "${out}"
python -c "import __graft_entry__ as g; g.build()" > "${out}/build.log" 2>&1 || { tail -20 "${out}/build.log"; exit 1; }
timeout 900 python -m pytest tests/test_gpu_finetune.py -m gpu -q -s > "${out}/finetune_tests.log" 2>&1; echo "finetune tests rc=$?"
grep "fine-tuning end to end" "${out}/finetune_tests.log"; tail -4 "${out}/finetune_tests.log"
timeout 2400 python -m pytest tests -m gpu -q --deselect tests/test_gpu_finetune.py > "${out}/gpu_suite.log" 2>&1; echo "gpu suite rc=$?"
tail -3 "${out}/gpu_suite.log"
timeout 300 python tools/time_finetune.py --steps 24 2>&1 | tee "${out}/time_finetune.log"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
timeout 300 python bench.py --gpus 1 --steps 200 --warmup 20 2>/dev/null | tail -1 > "${out}/bench.json"; head -c 400 "${out}/bench.json"; echo
