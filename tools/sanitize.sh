#!/bin/bash
# compute-sanitizer passes (memcheck, racecheck, synccheck) over one small invocation of every kernel (GPU box): once with the
# default solver policy (small batches: K2), once with the streamed solver forced
for mode in "default:" "streamed:PLSTVO_STREAM_SOLVE=1"; do
  name=${mode%%:*}; var=${mode#*:}
  for tool in memcheck racecheck synccheck; do
    echo "== $name / $tool"
    env $var compute-sanitizer --tool $tool --print-limit 5 python tools/sanitize_run.py 2>&1 | tail -6
  done
done
