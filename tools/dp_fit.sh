# Data parallelism through the model API: build, tests/test_gpu_dp_fit.py (two-device tests skip on fewer GPUs), the rest
# of the GPU suite, tools/time_fit_dp.py at N = 1, 2, 4, 8 (sizes above the device count are skipped), bench.py lines
# at the same N, smoke() and the default bench line.  Logs go to the directory given as the first argument (default: a
# fresh temporary directory).
set -u
out="${1:-$(mktemp -d)}"
mkdir -p "${out}"
python -c "import __graft_entry__ as g; g.build()" > "${out}/build.log" 2>&1 || { tail -20 "${out}/build.log"; exit 1; }
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader | tee "${out}/cards.txt"
timeout 900 python -m pytest tests/test_gpu_dp_fit.py -m gpu -q -rs > "${out}/dp_fit_tests.log" 2>&1; echo "dp fit tests rc=$?"
tail -6 "${out}/dp_fit_tests.log"
timeout 2400 python -m pytest tests -m gpu -q --deselect tests/test_gpu_dp_fit.py > "${out}/gpu_suite.log" 2>&1; echo "gpu suite rc=$?"
tail -3 "${out}/gpu_suite.log"
timeout 900 python tools/time_fit_dp.py --gpus 1 2 4 8 2>&1 | tee "${out}/time_fit_dp.log"
ngpu=$(nvidia-smi -L | wc -l)
for n in 1 2 4 8; do
  [ "${n}" -le "${ngpu}" ] || continue
  timeout 300 python bench.py --gpus "${n}" --steps 200 --warmup 20 2>/dev/null | tail -1 > "${out}/bench_n${n}.json"
  echo "bench N=${n}: $(head -c 300 "${out}/bench_n${n}.json")"
done
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
timeout 300 python bench.py --gpus 1 --steps 200 --warmup 20 2>/dev/null | tail -1 > "${out}/bench.json"; head -c 400 "${out}/bench.json"; echo
