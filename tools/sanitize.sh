#!/bin/bash
# compute-sanitizer over small parity tests of every kernel family (the team kernel synchronises
# through named barriers, shared-memory atomics and bulk async copies; the packed-expand and RLE
# kernels through warp-level primitives and bulk copies; the contour walk through __syncwarp around
# shared-memory updates of one lane).  Run on a GPU box:
#   bash tools/sanitize.sh   -> gpurun_out/sanitizer_<tool>.log
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
SEL="more_instances or every_box or no_detections or small_boxes or chunk_size or leading_unit or (packed_masks and (hw0 or hw1 or hw2 or hw7 or hw8)) or packed_batch_ragged or (rle_equals and not hw4 and not hw5) or rle_touching or all_zero_box or composite_on_device or out_of_range or alpha_sweep or (production_kernel and (small_mixed or tiny_boxes)) or identity_resize or byte_canvas_after or (contours_equal and float32 and (hw0 or hw2 or hw6 or hw7)) or hand_masks or boxes_limit or packed_and_canvas"
for tool in memcheck synccheck racecheck; do
  echo "== $tool"
  timeout 600 compute-sanitizer --tool $tool --error-exitcode 9 \
    python -m pytest tests/test_gpu_unmold.py tests/test_gpu_pack.py tests/test_gpu_rle.py tests/test_gpu_composite.py tests/test_gpu_contours.py \
    -q -x -k "$SEL" > gpurun_out/sanitizer_$tool.log 2>&1
  echo "exit $?"
  tail -3 gpurun_out/sanitizer_$tool.log
done
