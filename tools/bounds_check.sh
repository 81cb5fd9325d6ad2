# Builds libhmrm.so with -DHMRM_BOUNDS_CHECK (every table index of the traversal kernels validated on the device,
# compute-sanitizer is not available on the pool) and runs the GPU parity, fuzz and destination suites against it, then
# restores the production build.
set -e
HMRM_NVCC_EXTRA="-DHMRM_BOUNDS_CHECK" python heightmap-ray-marcher_b200/build.py --force > /dev/null 2>&1
python -m pytest tests/test_gpu_parity.py tests/test_gpu_fuzz.py tests/test_gpu_pyramid_fuzz.py \
	tests/test_gpu_destinations.py -m gpu -q 2>&1 | tail -4
python heightmap-ray-marcher_b200/build.py --force > /dev/null 2>&1
