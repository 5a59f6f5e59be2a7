#!/bin/bash
# quick GPU round trip: selected tests + timelines
set -u
mkdir -p gpurun_out
python -c "import __graft_entry__ as g; g.build()" > gpurun_out/build.log 2>&1 || { tail -20 gpurun_out/build.log; exit 1; }
timeout 900 python -X faulthandler -m pytest ${TESTS:-tests} -m gpu -q --maxfail=30 -p no:cacheprovider --timeout=300 > gpurun_out/pytest.log 2>&1; echo "pytest rc=$?"
tail -${TAILN:-15} gpurun_out/pytest.log
if [ "${TIMELINE:-0}" = "1" ]; then
SACB_TIMELINE=1 timeout 300 python tools/trace_stages.py > gpurun_out/trace_resident.log 2>&1
grep "timeline" gpurun_out/trace_resident.log | cut -c1-200
fi
