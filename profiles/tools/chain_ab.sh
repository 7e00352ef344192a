# A/B of ict_track_sequence: the whole chain in one K2v8 launch (default) against one launch per frame
timeout 600 python -m pytest tests/test_gpu_parity.py -q -x -k "chain or sequence or nposes" 2>&1 | tail -2
for s in 1 256 592 1184; do
echo "== $s chains, one launch";       SAMPLES=$s timeout 200 python profiles/tools/run_chain.py | tail -1
echo "== $s chains, launch per frame"; SEQ_LAUNCHES=1 SAMPLES=$s timeout 200 python profiles/tools/run_chain.py | tail -1
done
echo "== 592 chains donorm+patchnorm, one launch";       DONORM=1 PATCHNORM=1 SAMPLES=592 timeout 200 python profiles/tools/run_chain.py | tail -1
echo "== 592 chains donorm+patchnorm, launch per frame"; SEQ_LAUNCHES=1 DONORM=1 PATCHNORM=1 SAMPLES=592 timeout 200 python profiles/tools/run_chain.py | tail -1
