T="tests/test_blocks_gpu.py tests/test_unet_gpu.py::test_50_step_cfg_plms_sampling_cosine"
python -m pytest $T -x -q 2>&1 | grep -E "cosine|passed|failed"
