#!/bin/bash
# prioritized sampler after a change: bit-exactness tests, time per sample(256) at N = 1 M, adversarial sets
set -u
mkdir -p gpurun_out
timeout 900 python -X faulthandler -m pytest tests/test_gpu_replay.py -m gpu -q --maxfail=10 -p no:cacheprovider --timeout=300 > gpurun_out/pytest.log 2>&1; echo "pytest rc=$?"
grep -v "^\.\|^$\|^s" gpurun_out/pytest.log | tail -8 | cut -c1-300
python tools/per_profile.py 2>&1 | tail -3
python tools/per_adversarial.py 2>&1 | tail -3
