"""CPU-only tests: host logic, the C-ABI library's exported symbols, the NumPy Philox restatement,
and the world_size-2 gloo path of the episode-statistics all-gather.  No compute calls into CUDA."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import evac_testlib as T

ROOT = T.ROOT


def test_library_builds_and_exports_every_declared_symbol():
    from evacuation_b200 import _native as nat
    from evacuation_b200 import build as b

    path = b.build()
    assert os.path.exists(path)
    header = open(os.path.join(ROOT, "include", "evac_b200.h")).read()
    declared = set(re.findall(r"\b(evac_[a-z0-9_]+)\s*\(", header))
    assert declared == set(nat.SIGNATURES), declared ^ set(nat.SIGNATURES)
    lib = nat.load()  # binds every symbol; AttributeError if one is missing
    for name in declared:
        assert hasattr(lib, name)
    assert lib.evac_abi_version() == nat.EVAC_ABI_VERSION
    cfg = nat.EvacConfig()
    assert lib.evac_default_config(C.byref(cfg)) == 0
    # reference defaults: config.py:3-100, wrappers/config.py:8-44, constants.py:35-38
    assert (cfg.number_of_pedestrians, cfg.width, cfg.height, cfg.step_size, cfg.noise_coef, cfg.eps) == (10, 1.0, 1.0, 0.01, 0.2, 1e-8)
    assert (cfg.enslaving_degree, cfg.is_new_exiting_reward, cfg.is_new_followers_reward, cfg.intrinsic_reward_coef) == (1.0, 0, 1, 0.0)
    assert (cfg.init_reward_each_step, cfg.max_timesteps, cfg.alpha) == (-1.0, 2000, 3.0)
    assert (cfg.to_leader, cfg.to_pedestrian, cfg.to_exit, cfg.to_escape) == (0.2, 0.1, 0.4, 0.01)
    # the C struct layout seen by ctypes must match the compiler's: sizeof is checked through a NULL-handle call path
    assert lib.evac_obs_dim(None) == -1 and lib.evac_num_envs(None) == -1
    assert lib.evac_default_config(None) == -1 and b"NULL" in lib.evac_last_error()


def test_build_id_pins_the_binary_to_the_sources(tmp_path, monkeypatch):
    """Staleness is decided by content, not mtime: the library carries the SHA-256 of csrc/*.cu, csrc/*.cuh and
    include/*.h; a change to ANY of those files (evac_cluster.cuh was once missing from the header list) makes
    is_stale() true, and the loaded library reports the tree's hash."""
    import glob
    import shutil

    from evacuation_b200 import _native as nat
    from evacuation_b200 import build as b

    b.build()
    want = b.source_hash()
    assert re.fullmatch(r"[0-9a-f]{16}", want)
    assert b.library_build_id() == want and not b.is_stale()
    assert nat.load().evac_build_id().decode() == want == nat.build_id()
    tracked = {os.path.basename(p) for p in b.sources() + b.headers()}
    on_disk = {os.path.basename(p) for pat in ("csrc/*.cu", "csrc/*.cuh") for p in glob.glob(os.path.join(ROOT, "evacuation_b200", pat))}
    assert on_disk <= tracked and "evac_cluster.cuh" in tracked and "evac_b200.h" in tracked
    # a scratch copy of the tree: appending one byte to each file in turn changes the hash (mtimes play no role)
    csrc, inc = tmp_path / "csrc", tmp_path / "include"
    shutil.copytree(b.CSRC, csrc, ignore=shutil.ignore_patterns("*.o"))
    shutil.copytree(b.INCLUDE, inc)
    monkeypatch.setattr(b, "CSRC", str(csrc))
    monkeypatch.setattr(b, "INCLUDE", str(inc))
    assert b.source_hash() == want and not b.is_stale()
    for path in b.sources() + b.headers():
        old = open(path, "rb").read()
        with open(path, "ab") as f:
            f.write(b"\n")
        os.utime(path, (0, 0))  # an OLD mtime must not hide the change
        assert b.source_hash() != want and b.is_stale(), path
        open(path, "wb").write(old)
    assert b.source_hash() == want and not b.is_stale()


def test_cuda_library_contains_sm100a_packed_fp32_code():
    """The shipped .so carries sm_100a SASS with the packed FP32 pipe instructions of the pairwise pass."""
    from evacuation_b200 import build as b

    sass = subprocess.run(["cuobjdump", "-sass", b.build()], capture_output=True, text=True).stdout
    assert "sm_100a" in sass
    for op in ("FFMA2", "FADD2", "FMUL2", "FSET"):
        assert op in sass, op


def test_config_defaults_and_wrapper_dispatch_match_reference():
    import evacuation_b200 as eb

    c = eb.EnvConfig()
    assert (c.number_of_pedestrians, c.width, c.height, c.step_size, c.noise_coef, c.eps, c.enslaving_degree) == (10, 1.0, 1.0, 0.01, 0.2, 1e-8, 1.0)
    assert (c.is_new_exiting_reward, c.is_new_followers_reward, c.intrinsic_reward_coef, c.is_termination_agent_wall_collision) == (False, True, 0.0, False)
    assert (c.init_reward_each_step, c.max_timesteps, c.giff_freq, c.wandb_enabled) == (-1.0, 2000, 500, True)
    w = eb.EnvWrappersConfig()
    assert (w.num_obs_stacks, w.positions, w.statuses, w.type, w.alpha) == (1, "abs", "no", "Dict", 3)
    with pytest.raises(AssertionError):
        eb.EnvConfig(n_episodes=1)
    with pytest.raises(AssertionError):
        eb.EnvWrappersConfig(num_obs_stacks=4)
    with pytest.raises(NotImplementedError):
        eb.EnvWrappersConfig(positions="grav", type="Box").wrap_env(None)
    with pytest.raises(ValueError):
        eb.EnvWrappersConfig(positions="grav", type="Tuple").wrap_env(None)
    assert [s.value for s in eb.Status.all()] == [1, 2, 3, 4] and len(eb.Status) == 4
    assert (eb.SwitchDistances.to_leader, eb.SwitchDistances.to_pedestrian, eb.SwitchDistances.to_exit, eb.SwitchDistances.to_escape) == (0.2, 0.1, 0.4, 0.01)


def test_no_cpu_fallback():
    """Without a GPU the product path must fail loudly, never route through the oracle."""
    import torch

    import evacuation_b200 as eb
    from evacuation_b200._native import EvacNativeError

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(EvacNativeError):
        eb.setup_env(eb.EnvConfig(), eb.EnvWrappersConfig())
    src = "".join(open(os.path.join(ROOT, "evacuation_b200", f)).read() for f in os.listdir(os.path.join(ROOT, "evacuation_b200")) if f.endswith(".py"))
    assert "oracle" not in src.replace("never route through the oracle", "")


def test_spaces_and_agents():
    import evacuation_b200 as eb
    from evacuation_b200.spaces import Box

    box = Box(low=-1.0, high=1.0, shape=(2,), dtype=np.float32)
    a = eb.RandomAgent(box).act(None)
    assert a.dtype == np.float32 and a.shape == (2,) and box.contains(a)
    # the space samples from its own generator: the global MT19937 stream (which rng="numpy" retraces the reference with)
    # is left untouched, and seeding the space makes its samples reproducible (gymnasium semantics)
    np.random.seed(123)
    before = np.random.get_state()[1].copy(), np.random.get_state()[2]
    box.sample(); eb.RandomAgent(box).act(None)
    after = np.random.get_state()[1], np.random.get_state()[2]
    assert np.array_equal(before[0], after[0]) and before[1] == after[1]
    box.seed(7); s1 = box.sample(); box.seed(7)
    assert np.array_equal(s1, box.sample())
    r = eb.RotatingAgent(box)
    assert np.allclose(r.act(None), [np.sin(0.05), np.cos(0.05)]) and np.allclose(r.act(None), [np.sin(0.1), np.cos(0.1)])


def test_philox_known_answers():
    """Random123 known-answer vectors for Philox4x32-10 and Philox2x32-10."""
    kat = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
           ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
           ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0), (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]
    for ctr, key, want in kat:
        got = T.philox4x32_10(*ctr, *key)
        assert tuple(int(x) for x in got) == want
    for ctr, key, want in [((0, 0), 0, (0xFF1DAE59, 0x6CD10DF2)), ((0xFFFFFFFF, 0xFFFFFFFF), 0xFFFFFFFF, (0x2C3F628B, 0xAB4FD7AD)),
                           ((0x243F6A88, 0x85A308D3), 0x13198A2E, (0xDD7CE038, 0xF62A4C12))]:  # Random123 kat_vectors, philox2x32 10
        got = T.philox2x32_10(*ctr, key)
        assert (int(got[0]), int(got[1])) == want
    nz = T.philox_noise(7, 3, 1, 0, 60, 0.2)
    assert nz.dtype == np.float32 and np.all(np.abs(nz) <= 0.1) and len(np.unique(nz)) > 50


def test_noise_streams_do_not_alias_for_large_crowds(tmp_path):
    """ADVICE r1: with the block index OR-ed into the step field, pedestrian i + 4096 at step t drew pedestrian i's noise of
    step t + 1 (crowds above 4096).  (a) no two (pedestrian pair, step) tuples of one episode share a noise block any more;
    (b) the C++ stream (csrc/philox.cuh, compiled for the host) equals the NumPy restatement used by the parity tests."""
    n = 32768
    rows = np.stack([T.philox_noise(2024, 7, 3, now, n, 0.2) for now in (0, 1, 2, 7, 8, 15, 1999)])
    for r in rows:  # rows i and i + 4096 k differ within a step ...
        for k in range(1, 8):
            assert not np.array_equal(r[: n - 4096 * k], r[4096 * k:])
    flat = rows[:, ::1].reshape(len(rows), -1)
    for a in range(len(rows)):  # ... and no step is a shifted copy of another one
        for b_ in range(a + 1, len(rows)):
            for k in range(0, 8):
                assert not np.array_equal(flat[a][4096 * k: 4096 * k + 4096], flat[b_][:4096]), (a, b_, k)
    assert len(np.unique(rows[0])) > 0.99 * 2 ** 15 * (1 - 2 ** -10)  # 24-bit uniforms: almost no repeats among 32768 draws
    import shutil

    from evacuation_b200 import build as b

    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    src = tmp_path / "noise.cu"
    src.write_text('#include <cstdio>\n#include <cuda_runtime.h>\n#include "philox.cuh"\nusing namespace evac;\n'
                   "int main() { const unsigned nows[3] = {0u, 7u, 1999u};\n"
                   "  for (unsigned t = 0; t < 3; ++t) for (unsigned i = 0; i < 32768u; i += 61u) {\n"
                   "    const uint2 r = evac_noise_block(2024ull, 7u, 3u, nows[t], evac_noise_block_of(i));\n"
                   '    printf("%u %u %.9g\\n", nows[t], i, (double)((u01(evac_noise_word_of(i) ? r.y : r.x) - 0.5f) * 0.2f)); }\n'
                   "  return 0; }\n")
    exe = tmp_path / "noise"
    res = subprocess.run([nvcc, "-std=c++17", "-O1", "-I", b.CSRC, str(src), "-o", str(exe)], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    out = subprocess.run([str(exe)], capture_output=True, text=True).stdout.split()
    want = {0: T.philox_noise(2024, 7, 3, 0, n, 0.2), 7: T.philox_noise(2024, 7, 3, 7, n, 0.2), 1999: T.philox_noise(2024, 7, 3, 1999, n, 0.2)}
    vals = np.array(out, dtype=np.float64).reshape(-1, 3)
    assert len(vals) == 3 * len(range(0, 32768, 61))
    for now, i, v in vals:
        assert np.float32(v) == want[int(now)][int(i)], (now, i)


_POLICY_STREAM_PROGRAM = r"""
#include <cstdio>
#include "evac_policy.cuh"
using namespace evacp;
// record per (seed, offset, env, block, row): the words of every dropout site for d_model 2, 3, 6 ([attention | output] each)
// and F = 96 (hidden), then each word's dropped flag as the kernel decides it, at thresholds 6554 (p = 0.1) and 32768 (p = 0.5)
int main(int argc, char** argv) {
  FILE* f = fopen(argv[1], "wb");
  FILE* g = fopen(argv[2], "w");
  const unsigned long long seeds[2] = {0x2468ACE1ull, 0x13579BDF2468ACE1ull}, offs[3] = {0ull, 1ull, (1ull << 32) + 3ull};
  const uint32_t envs[4] = {0u, 5u, 65535u, (1u << 31) + 7u}, thr[2] = {6554u, 32768u};
  const int Ds[3] = {2, 3, 6};
  for (int s = 0; s < 2; ++s) for (int o = 0; o < 3; ++o) for (int e = 0; e < 4; ++e) {
    const uint32_t base = drop_base_key((uint32_t)seeds[s], (uint32_t)(seeds[s] >> 32), offs[o], envs[e]);
    for (int blk = 0; blk < 8; ++blk) for (int row = 0; row < 64; row += 2) {
      const uint32_t ka = drop_row_key(base, blk, row), kb = drop_row_key(base, blk, row + 1);  // a lane's two rows
      for (int r = 0; r < 2; ++r) {
        const uint32_t key = r ? kb : ka;
        uint16_t w[118];
        uint8_t m[2][118];
        int n = 0;
        for (int di = 0; di < 3; ++di)
          for (int site = 0; site < 2; ++site)
            for (int c = 0; c < Ds[di]; ++c, ++n) {
              w[n] = (uint16_t)drop_word(key, (uint32_t)(8 * site + c));
              for (int t = 0; t < 2; ++t) m[t][n] = w[n] < thr[t];
            }
        for (int fe = 0; fe < 96; ++fe, ++n) {
          const uint32_t t0a = drop_ff_word(ka, (uint32_t)(fe >> 2)), t0b = drop_ff_word(kb, (uint32_t)(fe >> 2));
          const uint2 t1 = drop_ff_mix(t0a, t0b);
          const uint32_t word = (fe & 2) ? (r ? t1.y : t1.x) : (r ? t0b : t0a);
          w[n] = (uint16_t)((fe & 1) ? word >> 16 : word & 0xFFFFu);
          for (int t = 0; t < 2; ++t) m[t][n] = drop_ff_dropped(word, fe & 1, thr[t] << 16);
        }
        fwrite(w, 2, 118, f);
        fwrite(m, 1, 236, f);
      }
    }
    // Normal draws of the heads (host libm: equal to float32 rounding, not bit for bit)
    const evac::Philox4 q = normal_words((uint32_t)seeds[s], (uint32_t)(seeds[s] >> 32), offs[o], envs[e]);
    const uint32_t words[4] = {q.x, q.y, q.z, q.w};
    fprintf(g, "%.9g %.9g %.9g\n", (double)normal_draw(words, 0), (double)normal_draw(words, 1), (double)normal_draw(words, 2));
  }
  fclose(f);
  fclose(g);
  return 0;
}
"""


def test_policy_streams_match_their_numpy_restatement(tmp_path):
    """The fused policy's dropout masks and Normal draws (csrc/evac_policy.cuh, compiled for the host) against the NumPy
    restatement in evac_testlib that the GPU tests of training mode build their float64 references from: every word of the
    attention, hidden (F = 96) and block-output sites for d_model 2 / 3 / 6, blocks 0..7, rows 0..63, seeds below and above 2^32,
    stream offsets 0, 1, 2^32 + 3 (the upper half enters the key) and global env indices 0, 5, 65535, 2^31 + 7, bit for bit,
    with the dropped flags at p = 0.1 and 0.5; and the three Box-Muller components of each (seed, offset, env)."""
    import shutil

    from evacuation_b200 import build as b

    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    src, exe = tmp_path / "streams.cu", tmp_path / "streams"
    src.write_text(_POLICY_STREAM_PROGRAM)
    res = subprocess.run([nvcc, "-std=c++17", "-O1", "-gencode", "arch=compute_100a,code=sm_100a", "-I", b.CSRC, str(src), "-o", str(exe)],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    words_path, normal_path = tmp_path / "words.bin", tmp_path / "normal.txt"
    subprocess.run([str(exe), str(words_path), str(normal_path)], check=True)
    raw = np.fromfile(words_path, dtype=np.uint8).reshape(2, 3, 4, 8, 64, 118 * 2 + 236)
    got_words = raw[..., :236].copy().view(np.uint16)
    got_flags = raw[..., 236:].reshape(raw.shape[:-1] + (2, 118))
    got_z = np.loadtxt(normal_path).reshape(2, 3, 4, 3)

    seeds, offs, envs = (0x2468ACE1, 0x13579BDF2468ACE1), (0, 1, 2 ** 32 + 3), (0, 5, 65535, 2 ** 31 + 7)
    blk, row = np.arange(8)[:, None], np.arange(64)[None, :]
    checked = 0
    for s, seed in enumerate(seeds):
        for o, off in enumerate(offs):
            for e, env in enumerate(envs):
                parts = []
                for D in (2, 3, 6):
                    attn, _, out = T.drop_site_words(seed, off, env, blk, row, D, 96)
                    parts += [attn, out]
                parts.append(T.drop_site_words(seed, off, env, blk, row, 6, 96)[1])
                want = np.concatenate(parts, axis=-1).astype(np.uint16)
                assert np.array_equal(got_words[s, o, e], want), (seed, off, env)
                for t, p in enumerate((0.1, 0.5)):
                    assert np.array_equal(got_flags[s, o, e, :, :, t], want < T.drop_threshold(p)), (seed, off, env, p)
                z, rad = T.policy_normal(seed, off, np.array([env]), 3)
                np.testing.assert_allclose(got_z[s, o, e], z[0], rtol=0, atol=2e-6 * (1 + rad[0].max()), err_msg=str((seed, off, env)))
                checked += 1
    assert checked == 24 and T.drop_threshold(0.1) == 6554 and T.drop_threshold(0.5) == 32768
    # the streams do move with every input: seeds, offsets (both halves), env index, block and row
    assert len({got_words[s, o, e, 0, 0].tobytes() for s in range(2) for o in range(3) for e in range(4)}) == 24
    assert len({got_words[0, 0, 0, b_, r].tobytes() for b_ in range(8) for r in range(64)}) == 512


def test_shard_partition():
    from evacuation_b200.distributed import shard_counts, shard_offset

    assert shard_counts(65536, 8) == [(i * 8192, 8192) for i in range(8)]
    parts = shard_counts(10, 4)
    assert parts == [(0, 3), (3, 3), (6, 2), (8, 2)] and sum(c for _, c in parts) == 10
    assert shard_offset(3, 4096) == 12288


_GLOO_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from evacuation_b200.distributed import allgather_totals_tensor, summarize_totals, shard_counts
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:" + sys.argv[2], rank=int(sys.argv[3]), world_size=2)
rank = dist.get_rank()
off, cnt = shard_counts(9, 2)[rank]
totals = torch.zeros(10, dtype=torch.float64)
totals[0] = cnt                      # "finished episodes" on this rank
totals[1:] = torch.arange(1, 10, dtype=torch.float64) * cnt * (rank + 1)
g = allgather_totals_tensor(totals)
assert g.shape == (2, 10) and g[0, 0] == 5 and g[1, 0] == 4, g
s = summarize_totals(g)
assert s["episodes"] == 9 and abs(s["episode_intrinsic_reward"] - (5 * 1 + 4 * 2) / 9) < 1e-12
dist.destroy_process_group()
print("ok", rank)
"""


def test_gloo_world_size_2_stats_allgather(tmp_path):
    import socket

    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = str(s.getsockname()[1])
    s.close()
    script = tmp_path / "w.py"
    script.write_text(_GLOO_WORKER)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, port, str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
             for r in range(2)]
    outs = [p.communicate(timeout=180)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0 and "ok" in o, o


def test_oracle_invariants_property():
    """SURVEY.md 8(a) invariants on the oracle: positions stay in the box, status is a pure function of the
    positions, ESCAPED is absorbing, rewards decompose."""
    from oracle.evac_oracle import ESCAPED, OracleConfig, OracleEnv, compute_statuses

    rs = np.random.RandomState(3)
    env = OracleEnv(OracleConfig(number_of_pedestrians=40, is_new_exiting_reward=True, intrinsic_reward_coef=0.7))
    np.random.seed(3)
    env.reset()
    escaped_before = np.zeros(40, bool)
    for t in range(400):
        _, r, term, trunc, info = env.step(np.array([0.2, -1.0], dtype=np.float32) + rs.uniform(-0.3, 0.3, 2).astype(np.float32))
        assert np.all(np.abs(env.positions) <= 1.0)
        st, _ = compute_statuses(env.positions, env.agent_position, env.exit_position)
        assert np.array_equal(st, env.statuses)
        assert np.all(env.statuses[escaped_before] == ESCAPED)
        escaped_before = env.statuses == ESCAPED
        assert r == info.reward_agent + info.reward_pedestrians + 0.7 * info.intrinsic_reward
        if term:
            break
    assert escaped_before.sum() > 0


def test_header_is_plain_c_and_the_library_is_a_c_abi():
    """include/evac_b200.h must compile as C99 (no torch / C++ types in the boundary) and a C program that only sees the
    header must link against libevac_b200.so and reach the entry points that need no GPU."""
    import shutil
    import tempfile

    from evacuation_b200 import build as b

    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    header = os.path.join(ROOT, "include", "evac_b200.h")
    res = subprocess.run([gcc, "-fsyntax-only", "-x", "c", "-std=c99", "-Wall", "-Werror", header], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    lib = b.build()
    with tempfile.TemporaryDirectory() as tmp:
        src = os.path.join(tmp, "t.c")
        with open(src, "w") as f:
            f.write('#include <stdio.h>\n#include "evac_b200.h"\n'
                    "int main(void) { EvacConfig c; if (evac_default_config(&c)) return 1;\n"
                    '  printf("%d %d %g\\n", (int)evac_abi_version(), (int)c.number_of_pedestrians, c.to_exit);\n'
                    "  return evac_default_config(0) == 0; }\n")
        exe = os.path.join(tmp, "t")
        res = subprocess.run([gcc, "-std=c99", "-I", os.path.join(ROOT, "include"), src, "-o", exe, lib, "-Wl,-rpath," + os.path.dirname(lib)],
                             capture_output=True, text=True)
        assert res.returncode == 0, res.stderr
        run = subprocess.run([exe], capture_output=True, text=True)
        assert run.returncode == 0, run.stderr
        version, n, to_exit = run.stdout.split()
        assert int(n) == 10 and float(to_exit) == 0.4 and int(version) >= 1


@pytest.mark.parametrize("force_port", [False, True])
def test_bench_reference_arm_prints_one_contract_line(force_port):
    """`bench.py --impl reference` (the reference's CPU step loop on the host cores; runs without a GPU): exactly one JSON line
    on stdout with the driver's keys, `impl`, a `cpu_baseline` describing the run and an `e2e` equal to the line's value.
    kind = "reference" (the unmodified reference through oracle/ref_shim.py) wherever a copy is reachable -- /root/reference
    here, baseline/_ref on the GPU box -- else "port" (the oracle)."""
    import json

    from oracle import ref_shim

    env = dict(os.environ, EVAC_BENCH_MIN_SECONDS="1")
    if force_port:
        env["EVAC_BENCH_CPU_KIND"] = "port"
    want_kind = "port" if force_port or not ref_shim.reference_available() else "reference"
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300, env=env)
    assert res.returncode == 0, res.stderr
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["impl"] == "reference" and d["steps"] == 3 and d["warmup"] == 1 and d["higher_is_better"] is True
    assert d["unit"] == "pedestrian-steps/s" and d["value"] > 0 and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == want_kind and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_bench_dump_outputs_are_float32_and_a_fixed_sample_under_64_mb(tmp_path):
    """`bench.py --dump-outputs`: one <name>.npy per array in float32 (flags as 0 / 1); above 64 MB in all, the same
    seeded sample of environments (ascending) is kept from every array, and the same one on every run."""
    import torch

    import bench

    E = 65536  # 65536 x (62 x 6 + 2) x 4 bytes = 98 MB
    arrays = {"obs": torch.rand((E, 62, 6), generator=torch.Generator().manual_seed(0)),
              "reward": torch.arange(E, dtype=torch.float32), "terminated": torch.arange(E) % 3 == 0}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["obs.npy", "reward.npy", "terminated.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 * 10 ** 6
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    rows = got["reward"].astype(np.int64)  # the reward column holds the environment index
    assert all(a.dtype == np.float32 and len(a) == len(rows) for a in got.values())
    assert E // 2 < len(rows) < E and np.all(np.diff(rows) > 0)
    np.testing.assert_array_equal(got["obs"], arrays["obs"].numpy()[rows])
    np.testing.assert_array_equal(got["terminated"], (rows % 3 == 0).astype(np.float32))
    for f in files:
        np.testing.assert_array_equal(np.load(tmp_path / "b" / f), got[f[:-4]])


def test_bind_host_to_device_never_raises():
    """The NUMA helper is opt-in plumbing for the host face: without NVML (this container) or on a single-node host it
    must report what it did and leave the process affinity usable."""
    from evacuation_b200.distributed import bind_host_to_device

    before = os.sched_getaffinity(0)
    info = bind_host_to_device(0)
    assert isinstance(info, dict) and "bound" in info
    after = os.sched_getaffinity(0)
    assert after and after <= before
    if not info["bound"]:
        assert after == before and "reason" in info


def test_renderer_draws_the_reference_scene(tmp_path):
    """SURVEY.md 8(f4): `render` / `save_animation` (env.py:173-324) rasterised with Pillow (matplotlib is absent from the
    image, so round 1's matplotlib code had never executed).  The scene is checked pixel-wise: pedestrians carry the
    status colours of matplotlib's default cycle in Status.all() order, the exiting zone is a green half disc ABOVE the exit,
    the following zone surrounds the agent, the GIF holds one 20 ms frame per recorded step."""
    from PIL import Image

    from evacuation_b200 import render as R

    pos = np.array([[0.5, 0.5], [-0.5, 0.5], [0.0, -0.8], [0.0, -1.0], [-0.7, -0.6]])
    st = np.array([1, 2, 3, 4, 1], dtype=np.uint8)
    img = R.draw_frame(pos, st, (0.3, 0.2), title="exp. Timesteps: 7")
    assert img.size == (R.SIZE, R.SIZE) and img.mode == "RGB"
    view = R._View(1.0, 1.0)

    def at(x, y):
        px, py = view.px(x, y)
        return img.getpixel((int(round(float(px))), int(round(float(py)))))

    assert at(0.5, 0.5) == R.STATUS_COLORS[1] and at(-0.5, 0.5) == R.STATUS_COLORS[2] and at(0.0, -0.8) == R.STATUS_COLORS[3]
    g = at(0.25, -0.9)           # inside the exiting zone (radius 0.4 around (0, -1), upper half): white blended with green at 0.2
    assert g[1] > g[0] and g[1] > g[2] and g != (255, 255, 255)
    assert at(0.25, -1.08) == (255, 255, 255)    # below the exit: outside the half disc
    b = at(0.3, 0.32)            # inside the following zone (radius 0.2 around the agent): white blended with blue at 0.1
    assert b[2] > b[0] and b[2] == 255 and b[0] < 255
    assert at(0.9, 0.9) == (255, 255, 255)
    png = R.save_png(str(tmp_path / "png" / "exp_7.png"), pos, st, (0.3, 0.2))
    assert Image.open(png).size == (R.SIZE, R.SIZE)
    T_ = 6
    traj = [pos + 0.01 * t for t in range(T_ + 1)]
    gif = R.save_gif(str(tmp_path / "giff" / "exp_ep-1.gif"), traj, [st] * (T_ + 1), [np.array([0.01 * t, 0.0]) for t in range(T_)], title="exp\nn_episodes = 1")
    im = Image.open(gif)
    assert im.n_frames == T_ and im.info.get("duration") == 20
    with pytest.raises(RuntimeError):
        R.save_gif(str(tmp_path / "x.gif"), [], [], [])
