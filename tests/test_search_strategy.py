"""The strategies bench.py loads ARE the reference Search Engine's output.  tests/golden/search_engine.json records one run of the
unmodified engine (galvatron/core/search_engine + csrc/dp_core.cpp, driven by scripts/search_strategy.py --memory-gb 178): the
profiles it was given and the strategy it returned at 1/2/4/8 GPUs.  The profiles must still be what scripts/search_strategy.py
and the committed B200 hardware tables produce, and configs/galvatron_config_llama3-8b_<N>gpus.json must be the engine's answer."""
import importlib.util
import json
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "search_engine.json")))
KEYS = ("pp_deg", "tp_sizes_enc", "tp_consecutive_flags", "dp_types_enc", "use_sp", "checkpoint", "global_bsz", "chunks", "pp_division",
        "pipeline_type", "default_dp_type", "vtp", "vsp", "embed_sdp")
HARDWARE = {"allreduce_bandwidth": "allreduce_bandwidth_1nodes_8gpus_per_node.json", "p2p_bandwidth": "p2p_bandwidth_1nodes_8gpus_per_node.json",
            "sp_time": "sp_time_1nodes_8gpus_per_node.json", "overlap_coefficient": "overlap_coefficient.json"}


def test_engine_inputs_are_what_the_search_script_produces():
    spec = importlib.util.spec_from_file_location("search_strategy", os.path.join(ROOT, "scripts", "search_strategy.py"))
    script = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(script)
    a = GOLD["profile_args"]
    time_cfg, mem_cfg = script.llama3_8b_profiles(a["layer_ms"], a["other_ms"], a["seq"])
    # through a JSON round trip: the engine read the profiles from files (string keys, floats as written)
    assert json.loads(json.dumps(time_cfg)) == GOLD["inputs"]["computation_profiling"]
    assert json.loads(json.dumps(mem_cfg)) == GOLD["inputs"]["memory_profiling"]
    for key, fname in HARDWARE.items():
        assert json.load(open(os.path.join(ROOT, "configs", "hardware_b200", fname))) == GOLD["inputs"][key], key


@pytest.mark.parametrize("n", [1, 2, 4, 8])
def test_bench_strategy_is_the_search_engines_output(n):
    got = GOLD["searched"][str(n)]
    want = json.load(open(os.path.join(ROOT, "configs", "galvatron_config_llama3-8b_%dgpus.json" % n)))
    for k in KEYS:
        if k in want or k in got:
            assert got.get(k) == want.get(k), (k, got.get(k), want.get(k))
    if n == 1:
        assert got["checkpoint"].split(",").count("1") == 15      # the engine's 20 % allocator reserve forces 15 of 32 layers
