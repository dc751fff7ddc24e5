#!/bin/bash
# GPU parity tests (selection via $1, e.g. "-k attention"); the log goes to $LOG_DIR (default test_logs/)
LOG_DIR=${LOG_DIR:-test_logs}
mkdir -p "$LOG_DIR"
timeout 600 python -m pytest tests/test_kernels_gpu.py tests/test_model_gpu.py tests/test_attention_exact_gpu.py -q --timeout 600 $1 > "$LOG_DIR/t_all.log" 2>&1; echo "tests exit $?"
grep -E "^E  |^FAILED|passed|failed" "$LOG_DIR/t_all.log" | cut -c1-400 | tail -40
