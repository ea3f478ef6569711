# Round-2 final measurements on one B200 (run under gpurun from the repo root); outputs under gpurun_out/final/.
# Every ncu pass follows a plain run of the same command (&&): a number printed under ncu is never a bench value.
mkdir -p gpurun_out/final
F=gpurun_out/final
python bench.py --steps 20 --warmup 5 > $F/bench_n1.json 2> $F/bench_n1.err
python bench.py --impl reference --steps 2 --warmup 1 > $F/bench_reference_arm.json 2> $F/bench_reference_arm.err
python profiles/measure_configs.py > $F/config_timings.json 2> $F/config_timings.err
python profiles/measure_build.py > $F/build_timings.json 2> $F/build_timings.err
python profiles/measure_reduce_profile.py > $F/reduce_profile.json 2> $F/reduce_profile.err
SWEEPS=1720 BEAMS=1744 python profiles/measure_reduce_profile.py > $F/reduce_profile_3M.json 2> $F/reduce_profile_3M.err
python profiles/measure_sequence.py > $F/sequence.json 2> $F/sequence.err
python profiles/measure_normals.py > $F/normals_depth.json 2> $F/normals_depth.err
python profiles/probe_pair_queue.py > $F/pair_queue_contexts.txt 2> $F/pair_queue_contexts.err
python profiles/probe_sequence_frame.py > $F/sequence_frame_breakdown.json 2> $F/sequence_frame_breakdown.err
# the 44-pair queue replayed on one GPU (every pair alone, every rank's share of the static deals), why the pairs differ in cost,
# and the group search: A/B of the bench line and the configs, per pair with the diagnostic counters, on a point shard
python profiles/probe_pair_queue_deal.py > $F/pair_queue_deal_probe.json 2> $F/pair_queue_deal_probe.err
python profiles/probe_pair_costs.py > $F/pair_costs_by_distance.json 2> $F/pair_costs_by_distance.err
bash profiles/ab_group.sh > $F/group_search_ab.txt 2>&1
make -C icp_variants_b200/csrc groupprobe > $F/make_groupprobe.log 2>&1
ICP_GPU_LIB_NAME=libicp_gpu_groupprobe.so PAIRS=0,28,34 GROUP_MINS="0 8" python profiles/probe_group.py > $F/group_search_per_pair.json 2> $F/group_search_per_pair.err
rm -f icp_variants_b200/lib/libicp_gpu_groupprobe.so icp_variants_b200/lib/knn_groupprobe.o
python profiles/probe_group_shard.py > $F/group_search_on_a_shard.json 2> $F/group_search_on_a_shard.err
# per-warp timeline of one iteration, one and two chunk chains (diagnostic build of the library, removed again afterwards)
make -C icp_variants_b200/csrc timeline > $F/make_timeline.log 2>&1
ICP_GPU_MATCH_CHUNKS=1 python profiles/probe_timeline.py > $F/timeline_1chunk.json 2> $F/timeline_1chunk.err
ICP_GPU_MATCH_CHUNKS=2 python profiles/probe_timeline.py > $F/timeline_2chunks.json 2> $F/timeline_2chunks.err
rm -f icp_variants_b200/lib/libicp_gpu_timeline.so icp_variants_b200/lib/*_timeline.o
B="python bench.py --steps 2 --warmup 3 --no-cpu-baseline --no-multi"
# launch lists of the bench command: caches as the program leaves them (--cache-control none: the figures that add up to the step),
# and ncu's default (flushed before every launch: cold-cache, compare shares only)
$B > $F/plain.log 2>&1 && ncu --metrics gpu__time_duration.sum --cache-control none --clock-control none -c 700 --csv --log-file $F/launches_hot.csv $B > $F/ncu_launches_hot.log 2>&1
$B > $F/plain.log 2>&1 && ncu --metrics gpu__time_duration.sum --clock-control none -c 700 --csv --log-file $F/launches.csv $B > $F/ncu_launches.log 2>&1
# one full capture of the iteration kernels (a steady-state iteration) and of the index-build kernels; the iteration kernels with ONE
# chunk chain (ICP_GPU_MATCH_CHUNKS=1), so that a launch covers all queries like the launches bench.py's roofline object times
export ICP_GPU_MATCH_CHUNKS=1
$B > $F/plain.log 2>&1 && ncu --set full --clock-control none --import-source on -k regex:"knn_prep|knn_group|knn_bvh|reduce_kernel" -s 400 -c 4 -f -o $F/prof_hot $B > $F/ncu_full.log 2>&1
unset ICP_GPU_MATCH_CHUNKS
python profiles/measure_build.py > $F/plain_build.log 2>&1 && ncu --set full --clock-control none --cache-control none --import-source on -k regex:"pack_bbox|keys_kernel|radix_|gather_records|level_|bvh_level|upper_levels|leaf_adjacency|seed_from_keys" -s 60 -c 24 -f -o $F/prof_build python profiles/measure_build.py > $F/ncu_build.log 2>&1
python profiles/profile_projective.py > $F/plain_proj.log 2>&1 && ncu --set full --clock-control none --cache-control none --import-source on -k regex:projective -s 40 -c 1 -f -o $F/prof_proj python profiles/profile_projective.py > $F/ncu_proj.log 2>&1
tail -c 400 $F/bench_n1.json
