"""Runs the reference's own C kernels (lance-linalg/src/simd/f16.c and dist_table.c, compiled into
oracle/_ref/libref_simd.so by `make -C oracle ref REF=<reference checkout>/rust/lance-linalg/src/simd`) on
fixed inputs and stores inputs and outputs as tests/golden/ref_simd_outputs.npz, so that
tests/test_oracle_golden.py compares the oracle with the reference kernels without the reference sources.
Nothing here is computed by our code.  Run:  python tests/golden/make_ref_simd_outputs.py
"""
import ctypes as C
import json
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
so = os.path.join(os.path.dirname(os.path.dirname(HERE)), "oracle", "_ref", "libref_simd.so")
ref = C.CDLL(so)
ref.l2_f16_avx2.restype = C.c_float
ref.l2_f16_avx2.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
ref.sum_4bit_dist_table_32bytes_batch_avx512.restype = None
ref.sum_4bit_dist_table_32bytes_batch_avx512.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]

out = {}
# l2_f16_avx2, built -ffast-math as lance-linalg/build.rs:99 does
dims = (8, 16, 128, 130, 768)
rng = np.random.default_rng(1)
for d in dims:
    x = rng.standard_normal(d).astype(np.float16)
    y = rng.standard_normal(d).astype(np.float16)
    out[f"f16_x_{d}"], out[f"f16_y_{d}"] = x, y
    out[f"f16_l2_{d}"] = np.float32(ref.l2_f16_avx2(x.ctypes.data, y.ctypes.data, d))
out["f16_dims"] = np.array(dims, np.int64)

# sum_4bit_dist_table_32bytes_batch_avx512 (dist_table.c:8): the reference's known-answer literal (dist_table.rs:179-217)
# and random codes; the kernel consumes 64 code bytes (= 2 sub-vector pairs) per step
cases = json.load(open(os.path.join(HERE, "reference_known_answers.json")))
dt = [(np.asarray(c["codes"], np.uint8), np.asarray(c["dist_table"], np.uint8), c["code_len"])
      for c in cases if c["op"] == "sum_4bit_dist_table"]
rng = np.random.default_rng(7)
for code_len in (2, 4, 8, 16):
    dt.append((rng.integers(0, 256, 32 * code_len, dtype=np.uint8),
               rng.integers(0, 256 // (2 * code_len), 32 * code_len, dtype=np.uint8), code_len))
for i, (codes, table, code_len) in enumerate(dt):
    res = np.zeros(32, np.uint16)
    ref.sum_4bit_dist_table_32bytes_batch_avx512(codes.ctypes.data, codes.size, table.ctypes.data, res.ctypes.data)
    out[f"dt_codes_{i}"], out[f"dt_table_{i}"], out[f"dt_code_len_{i}"], out[f"dt_sum_{i}"] = codes, table, code_len, res
out["dt_cases"] = len(dt)

path = os.path.join(HERE, "ref_simd_outputs.npz")
np.savez_compressed(path, **out)
print("wrote", path, os.path.getsize(path), "bytes")
