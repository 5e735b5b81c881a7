#!/bin/bash
# the model-level GPU tests with each fast path switched off in turn (the model tests use the dense paths as references; every
# combination has to stay correct)
for e in RBM_SAS_LIVE_ROWS=0 RBM_BERT_LABEL_ROWS=0 RBM_BERT_LABEL_QUERIES=0; do
  echo "== $e"
  env $e timeout 900 python -m pytest tests/test_models_gpu.py -m gpu -q -x 2>&1 | tail -1 | cut -c1-200
done
# the attention tests with every dense call on the SIMT kernels (the library reads the switch once per process: one process per setting)
echo "== RBM_ATTN_IMPL=mma"
env RBM_ATTN_IMPL=mma timeout 900 python -m pytest tests/test_attention_gpu.py tests/test_kernels_gpu.py -k attention -m gpu -q -x 2>&1 | tail -1 | cut -c1-200
