"""The CPU restatement of the production random numbers (`tests/philox_model.py`) against the Philox4x32-10
definition (Random123 known answers) and against `csrc/philox.cuh` itself, compiled for the host."""

import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

from tests import philox_model as pm

ROOT = Path(__file__).resolve().parent.parent
CSRC = ROOT / "attpc_engine_b200" / "csrc"


@pytest.mark.parametrize(
    "ctr, key, want",
    [
        ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
        ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
        ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
         (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
    ],
    ids=["zero", "ones", "pi"],
)  # fmt: skip
def test_random123_known_answers(ctr, key, want):
    got = pm.philox4x32_10(*ctr, *key)
    assert tuple(int(w) for w in got) == want


_HOST_SRC = r"""
#include <cstdio>
#include <vector>
#include "philox.cuh"
// stdin: n, then n x (c0 c1 c2 c3 k0 k1) as uint32; stdout: n x (x0 x1 x2 x3 as uint32, uniform, uniform16 as double)
int main() {
    long long n = 0;
    if (fread(&n, sizeof n, 1, stdin) != 1) return 1;
    std::vector<uint32_t> in(6 * n);
    if ((long long)fread(in.data(), 4, 6 * n, stdin) != 6 * n) return 1;
    for (long long i = 0; i < n; ++i) {
        const uint32_t* c = &in[6 * i];
        const attpc::Philox4 r = attpc::philox4x32_10(c[0], c[1], c[2], c[3], c[4], c[5]);
        const uint64_t ev = ((uint64_t)c[1] << 32) | c[0], seed = ((uint64_t)c[5] << 32) | c[4];
        const double u = attpc::philox_uniform(seed, ev, c[2], c[3]), u16 = attpc::philox_uniform16(seed, ev, c[2], c[3]);
        const uint32_t w[4] = {r.x, r.y, r.z, r.w};
        fwrite(w, 4, 4, stdout);
        fwrite(&u, 8, 1, stdout);
        fwrite(&u16, 8, 1, stdout);
    }
    return 0;
}
"""


def _counters(n=100_000):
    rng = np.random.default_rng(20261020)
    words = rng.integers(0, 2**32, size=(n, 6), dtype=np.uint64).astype(np.uint32)
    words[-1000:, 2] = pm.STREAM_WIGGLE
    edge = np.array([0, 1, 0x7FFFFFFF, 0x80000000, 0xFFFFFFFF], dtype=np.uint32)
    # every edge word in every position (with random others), and every position at all-edges
    rows = []
    for pos in range(6):
        for v in edge:
            r = rng.integers(0, 2**32, size=6, dtype=np.uint64).astype(np.uint32)
            r[pos] = v
            rows.append(r)
    for v in edge:
        rows.append(np.full(6, v, dtype=np.uint32))
    return np.concatenate([words, np.array(rows, dtype=np.uint32)])


def test_restatement_matches_the_header_bit_for_bit(tmp_path):
    nvcc = shutil.which("nvcc") or (shutil.which("nvcc", path="/usr/local/cuda/bin"))
    if nvcc is None:
        pytest.skip("nvcc is not installed")
    src = tmp_path / "philox_host.cu"
    src.write_text(_HOST_SRC)
    exe = tmp_path / "philox_host"
    cmd = [nvcc, "-Wno-deprecated-gpu-targets", "-std=c++17", "-O2", "-I", str(CSRC), "-o", str(exe), str(src)]
    subprocess.run(cmd, check=True)
    c = _counters()
    stdin = np.array([len(c)], dtype=np.int64).tobytes() + c.tobytes()
    out = subprocess.run([str(exe)], input=stdin, capture_output=True, check=True).stdout
    rec = np.frombuffer(out, dtype=np.dtype([("w", "<u4", 4), ("u", "<f8"), ("u16", "<f8")]))
    assert len(rec) == len(c)
    got = np.stack(pm.philox4x32_10(*c.T), axis=1)
    assert np.array_equal(got, rec["w"])
    seed = (c[:, 5].astype(np.uint64) << np.uint64(32)) | c[:, 4]
    event = (c[:, 1].astype(np.uint64) << np.uint64(32)) | c[:, 0]
    assert np.array_equal(pm.philox_uniform(seed, event, c[:, 2], c[:, 3]), rec["u"])
    assert np.array_equal(pm.philox_uniform16(seed, event, c[:, 2], c[:, 3]), rec["u16"])
    # the wiggle is the 16-bit uniform of stream 0xFFFFFFFF
    m = c[:, 2] == pm.STREAM_WIGGLE
    assert m.sum() >= 1000
    assert np.array_equal(pm.wiggle16(seed[m], event[m], c[m, 3]), rec["u16"][m])


def test_counter_layout_uses_both_words_of_event_and_seed():
    """Each of the six counter/key words reaches the output (no word is dropped or aliased)."""
    base = pm.fano_normal(7, 5, 3, 11)[0]
    assert pm.fano_normal(7, 5 + 2**32, 3, 11)[0] != base
    assert pm.fano_normal(7 + 2**32, 5, 3, 11)[0] != base
    assert pm.fano_normal(7, 5, 4, 11)[0] != base
    assert pm.fano_normal(7, 5, 3, 12)[0] != base
    x = pm.philox4x32_10(5, 0, 3, 11, 7, 0)
    assert pm.fano_normal(7, 5, 3, 11)[0] == pm.box_muller(pm.uniform53(x[0], x[1]), x[2])[0]
    assert pm.wiggle16(7, 5, 99) == (int(pm.philox4x32_10(5, 0, 0xFFFFFFFF, 99, 7, 0)[0]) >> 16) / 65536.0


def test_box_muller_extremes_keep_the_gate_exact():
    """|z| is largest at u53 = 0 (u1 = 2^-54) and zero at u53 = 1 - 2^-53 (u1 rounds to 1): with the error bound of
    the device's float32 evaluation it stays below NORMAL_ABS_MAX, so mean + spread * NORMAL_ABS_MAX < 1 means no
    electron whatever the draw."""
    u53 = np.array([0.0, 1.0 - 2.0**-53])
    for x2 in (0, 0xFFFFFFFF, 0x80000000, 0x40000000):  # cos(2 pi u2) = 1, ~1, -1, ~0
        z, err = pm.box_muller(u53, np.full(2, x2, dtype=np.uint32))
        assert np.all(np.abs(z) + err < pm.NORMAL_ABS_MAX)
    z, err = pm.box_muller(u53, np.zeros(2, dtype=np.uint32))
    assert z[0] == pytest.approx(np.sqrt(108.0 * np.log(2.0)), rel=1e-15) and z[1] == 0.0
    assert 8.65 < z[0] + err[0] < pm.NORMAL_ABS_MAX


def test_normals_are_standard():
    z, err = pm.fano_normal(11, np.arange(200_000), 2, 5)
    assert abs(z.mean()) < 0.01 and abs(z.std() - 1.0) < 0.01
    assert np.all(err < 1e-5)
