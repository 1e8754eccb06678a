#!/bin/bash
# compute-sanitizer over a subset of the GPU tests that covers every kernel family with hand-rolled synchronisation:
# mbarrier rings + cp.async.bulk (RoIAlign tile / window kernels), tensor-memory alloc / ld / st (RoIAlign backward,
# overlap, scoring), cp.async private slots + tcgen05.mma (overlap), TMA + tcgen05 (scoring fwd / bwd), the mining
# kernels' shared-memory sorts, the loss block.  Logs -> gpurun_out/ (summaries are committed under profiles/).
#   gpurun --timeout 1500 -- 'bash tools/sanitize.sh'
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
SEL='tile_path_small or window_tiles_match_oracle or maskfuse_tile_path or tensor_core_kernel_repeated_launches or backward_tile_in_tensor_memory or sparse_crop_unpack or fused_crop_unpack or score_heads_reference_fixture or score_heads_backward_tensor or reference_fixtures or device_anti_noise or step_matches_oracle or test_box_nms or roi_pool_tile_kernels_equal or stream_sampling or batched_matches_oracle or (native_image_sizes and n300) or (tile_geometry_sweep and one_image)'
for tool in memcheck racecheck; do
  timeout 1200 compute-sanitizer --tool $tool --error-exitcode 0 --print-limit 20 \
      python -m pytest tests -m gpu -q -x -k "$SEL" -p no:cacheprovider > gpurun_out/sanitizer_$tool.log 2>&1
  echo "== $tool: exit $?"; grep -E "ERROR SUMMARY|RACECHECK SUMMARY|passed|failed|error" gpurun_out/sanitizer_$tool.log | tail -5
done
