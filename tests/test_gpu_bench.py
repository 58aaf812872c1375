"""bench.py --dump-outputs on a small synthetic workload: the logits and recurrent state it writes must be exactly what the library
computes for the token stream the timed path evaluated, and --steps must set how many timed steps that stream holds."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu
PRESET, FMT, WARMUP, CHUNK = "rwkv6-small", "Q5_1", 3, 128


@pytest.mark.parametrize("mode", ["decode", "prefill"])
def test_dump_outputs_are_the_last_timed_step(pkg, lib, tmp_path, mode):
    import synthetic_model as sm
    env = dict(os.environ, RWKV_B200_BENCH_DIR=str(tmp_path))
    path = str(tmp_path / f"{PRESET}-{FMT}-seed1.bin")
    dumps = {}
    for steps in (2, 3):
        out = tmp_path / f"dump-{steps}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", f"{PRESET}:{FMT}", "--mode", mode, "--steps", str(steps),
                            "--warmup", str(WARMUP), "--prefill-steps", "1", "--skip-cpu-baseline", "--dump-outputs", str(out)],
                           capture_output=True, text=True, env=env, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        assert sorted(os.listdir(out)) == ["logits.npy", "state.npy"]
        dumps[steps] = [np.load(out / "logits.npy"), np.load(out / "state.npy")]
        assert all(a.dtype == np.float32 for a in dumps[steps])
    assert not np.array_equal(dumps[2][1], dumps[3][1])
    model = pkg.RWKVModel(lib, path, thread_count=1)
    try:
        for steps, (logits, state) in dumps.items():
            if mode == "decode":    # one untimed token allocates the buffers, then warm-up and timed steps start over from token 0
                toks = sm.synthetic_tokens(WARMUP + steps, model.n_vocab)
                want_logits, want_state = model.eval(toks[0], None, use_numpy=True)
                for t in toks:
                    want_logits, want_state = model.eval(t, want_state, use_numpy=True)
            else:                   # fresh state, warm-up and timed chunks of 128 tokens
                toks = sm.synthetic_tokens(CHUNK * (WARMUP + steps), model.n_vocab)
                want_logits, want_state = model.eval_sequence_in_chunks(toks, None, chunk_size=CHUNK, use_numpy=True)
            assert np.array_equal(logits, want_logits), (mode, steps)
            assert np.array_equal(state, want_state), (mode, steps)
    finally:
        model.free()
