# Group saliency maps: build, the group-saliency GPU tests, tools/time_group_saliency.py (schedules and the end-to-end
# call, then k_group_colsum under torch.profiler in a run of its own), the rest of the GPU suite, smoke() and one bench
# line.  Logs go to the directory given as the first argument (default: a fresh temporary directory).
set -u
out="${1:-$(mktemp -d)}"
mkdir -p "${out}"
python -c "import __graft_entry__ as g; g.build()" > "${out}/build.log" 2>&1 || { tail -20 "${out}/build.log"; exit 1; }
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "${out}/card.txt"
timeout 1500 python -m pytest tests/test_gpu_group_saliency.py -m gpu -q -x > "${out}/group_saliency_tests.log" 2>&1
echo "group saliency tests rc=$?"
tail -30 "${out}/group_saliency_tests.log"
timeout 600 python tools/time_group_saliency.py --steps 20 2>&1 | tee "${out}/time_group_saliency.log"
timeout 300 python tools/time_group_saliency.py --steps 20 --profile 2>&1 | tee "${out}/profile_group_saliency.log"
timeout 2400 python -m pytest tests -m gpu -q --deselect tests/test_gpu_group_saliency.py > "${out}/gpu_suite.log" 2>&1
echo "gpu suite rc=$?"
tail -3 "${out}/gpu_suite.log"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
timeout 300 python bench.py --gpus 1 --steps 200 --warmup 20 2>/dev/null | tail -1 > "${out}/bench.json"; head -c 400 "${out}/bench.json"; echo
