#!/bin/bash
# A/B of source trees on one box: the working tree vs other trees (default .ab_head, a build of HEAD).
# Usage: gpurun --timeout 600 -- 'bash tools/ab_trees.sh TAG [OTHER_TREE ...]'
TAG=${1:-x}; shift; OTHERS=${@:-.ab_head}
mkdir -p gpurun_out
{
for rep in 1 2; do
  echo "== decoder, tree=new";   python tools/decoder_ab.py
  for o in $OTHERS; do echo "== decoder, tree=$o"; LAS_ROOT=$PWD/$o python tools/decoder_ab.py; done
  echo "== listener, tree=new";   python tools/listener_ab.py
  for o in $OTHERS; do echo "== listener, tree=$o"; LAS_ROOT=$PWD/$o python tools/listener_ab.py; done
done
} > gpurun_out/ab_$TAG.log 2>&1
cat gpurun_out/ab_$TAG.log
