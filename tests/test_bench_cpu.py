"""CPU: what bench.py --dump-outputs writes (whole outputs, or a sample at positions fixed by the output's name) and the
argument checks that run before any GPU work."""
import subprocess
import sys

import torch

import bench


def test_dump_sample_is_whole_or_a_fixed_sample():
    small = torch.arange(12.0, dtype=torch.float64).reshape(3, 4)
    out = bench.dump_sample(small, "latents")
    assert out.dtype == torch.float32 and torch.equal(out, small.float())
    big = torch.randn(bench.DUMP_MAX_ELEMENTS + 1000)
    a, b = bench.dump_sample(big, "vae_decode_frames"), bench.dump_sample(big.clone(), "vae_decode_frames")
    assert a.dtype == torch.float32 and a.shape == (bench.DUMP_MAX_ELEMENTS,) and torch.equal(a, b)
    assert not torch.equal(a, bench.dump_sample(big, "vae_encode_latents"))


def test_bench_rejects_bad_arguments():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        r = subprocess.run([sys.executable, bench.__file__, *extra], capture_output=True, text=True, timeout=300)
        assert r.returncode == 2 and "error:" in r.stderr, (extra, r.stderr[-500:])
