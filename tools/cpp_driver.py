"""Shared helpers for running the COMPILED proof driver (include/spectre_b200_prover.hpp via tests/cpp/prover_main.cpp)
against libspectre_b200.so: build the binary, dump a circuit instance in the format prover_main reads, run it.
Used by tests/test_cpp_prover.py (parity) and bench.py (timing next to the Python driver). No oracle involved."""
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def build_main_against_the_real_library(out_dir=None):
    """g++ tests/cpp/prover_main.cpp -DSPB_PROVER_WITH_CUDART against libspectre_b200.so + cudart -> prover_main_cuda in
    out_dir (default tests/cpp/)"""
    from spectre_b200 import build
    lib = build.build()
    libdir = os.path.dirname(lib)
    exe = os.path.join(out_dir or os.path.join(ROOT, "tests", "cpp"), "prover_main_cuda")
    src = os.path.join(ROOT, "tests", "cpp", "prover_main.cpp")
    hdrs = [os.path.join(ROOT, "include", h) for h in ("spectre_b200.h", "spectre_b200_prover.hpp")]
    if os.path.exists(exe) and os.path.getmtime(exe) >= max(os.path.getmtime(p) for p in [src, lib] + hdrs):
        return exe
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-DSPB_PROVER_WITH_CUDART", "-I" + os.path.join(cuda, "include"), "-o", exe, src,
                           "-L" + libdir, "-lspectre_b200", "-Wl,-rpath," + libdir, "-L" + os.path.join(cuda, "lib64"), "-lcudart",
                           "-Wl,-rpath," + os.path.join(cuda, "lib64")])
    return exe


def dump_case(d, head, k, digest, instances, copies, rng_counts, fixed, adv, rng_rows, tau, chacha_poly=None):
    """head: 'shape aggregation' | 'shape halo2lib G L'; rng_counts: create_proof's draw sizes in order (zeros included);
    rng_rows: the drawn rows for the non-zero counts, in order; tau: (4,) uint64 Montgomery SRS secret; chacha_poly: 32-byte
    seed when the vanishing argument's random polynomial comes from the device ChaCha20 stream (that draw is then absent
    from rng_counts / rng_rows)."""
    with open(os.path.join(d, "meta.txt"), "w") as f:
        f.write(head + "\nk %d\ndigest %x\ninstances %s\n" % (k, digest, " ".join("%x" % v for v in instances)))
        for (c1, r1), (c2, r2) in copies:
            f.write("copy %d %d %d %d\n" % (c1, r1, c2, r2))
        f.write("rng " + " ".join(str(c) for c in rng_counts) + "\n")
        if chacha_poly is not None:
            f.write("chacha_poly %s\n" % bytes(chacha_poly).hex())
    with open(os.path.join(d, "fixed.bin"), "wb") as f:
        for c in fixed:
            f.write(np.ascontiguousarray(c, dtype=np.uint64).tobytes())
    with open(os.path.join(d, "advice.bin"), "wb") as f:
        for c in adv:
            f.write(np.ascontiguousarray(c, dtype=np.uint64).tobytes())
    with open(os.path.join(d, "rng.bin"), "wb") as f:
        for rows in rng_rows:
            f.write(np.ascontiguousarray(rows, dtype=np.uint64).tobytes())
    np.ascontiguousarray(tau, dtype=np.uint64).reshape(4).tofile(os.path.join(d, "tau.bin"))


def run(exe, d, repeat=1, tables=False, timeout=900):
    """-> (returncode, stdout+stderr, proof bytes or None, [create_proof_ms...], keygen_ms or None)"""
    env = dict(os.environ, SPB_MAIN_REPEAT=str(repeat))
    if tables:
        env["SPB_MAIN_TABLES"] = "1"
    out = subprocess.run([exe, d], capture_output=True, text=True, env=env, timeout=timeout)
    proof = None
    if out.returncode == 0:
        with open(os.path.join(d, "proof.bin"), "rb") as f:
            proof = f.read()
    ms = [float(l.split()[1]) for l in out.stdout.splitlines() if l.startswith("create_proof_ms")]
    kg = [float(l.split()[1]) for l in out.stdout.splitlines() if l.startswith("keygen_ms")]
    return out.returncode, out.stdout + out.stderr, proof, ms, (kg[0] if kg else None)


class RecordingRng:
    """wraps an rng(count) -> (count, 4) callable and keeps every draw, so the compiled driver can replay the same stream"""

    def __init__(self, inner, chacha_poly=None):
        """chacha_poly: 32-byte seed -> the bulk draw (the random polynomial) is made in device memory by the engine from that
        ChaCha20 stream (rng.device_rows protocol of plonk.create_proof) and is not part of the recorded host stream"""
        self.inner, self.calls, self.chacha_poly = inner, [], chacha_poly
        if chacha_poly is not None:
            self.device_rows = lambda E, count: E.random_chacha(bytes(chacha_poly), 0, count)

    def __call__(self, count):
        out = self.inner(count)
        self.calls.append(np.ascontiguousarray(out, dtype=np.uint64).reshape(-1, 4))
        return out

    @property
    def counts(self):
        return [c.shape[0] for c in self.calls]

    @property
    def rows(self):
        return [c for c in self.calls if c.shape[0]]
