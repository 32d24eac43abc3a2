"""Run the SIMT kernels of csrc/roc.cu and csrc/bce_head.cu on the CPU under a small CUDA execution-model emulator
(tests/emu/cuda_emu.h: one fiber per CUDA thread, rendezvous at __syncthreads / __shfl) and compare with the oracles.

This checks the kernels' indexing, tiling, barrier placement and reductions without a GPU (the GPU parity tests remain
the authority on the real hardware path).  The kernel source is taken verbatim from the .cu file up to the end of its
``namespace pfc`` block; only the ``#include "common.cuh"`` line is replaced by the emulator header."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

# EMU_ASAN=1 (set by test_emulated_kernels_under_address_sanitizer for its child process) instruments the emulated builds
SAN_FLAGS = ["-fsanitize=address", "-fno-omit-frame-pointer", "-g"] if os.environ.get("EMU_ASAN") == "1" else []

HARNESS = {
    "roc": r'''
extern "C" void emu_roc(const float* feature, const int32_t* label, int64_t n, const float* sub, const int32_t* sublabel,
                        int64_t n_sub, int64_t sub_offset, int emb, unsigned long long* hist, int grid) {
  emu_launch((unsigned)grid, pfc::kRocThreads, [=]() {
    pfc::roc_hist_kernel(feature, label, n, sub, sublabel, n_sub, sub_offset, emb, hist);
  });
}
''',
    "roc2": r'''
extern "C" void emu_roc2(const float* feature, const int32_t* label, int64_t n, const float* sub, const int32_t* sublabel,
                         int64_t n_sub, int64_t sub_offset, int emb, float coef, unsigned long long* hist, int grid) {
  emu_launch((unsigned)grid, pfc::kRocThreads, [=]() {
    pfc::roc_hist2_kernel(feature, label, n, sub, sublabel, n_sub, sub_offset, emb, coef, hist);
  });
}
''',
    "hardneg": r'''
extern "C" void emu_similar(const float* a, int64_t n_a, const float* b, int64_t n_b, int emb, float thr, unsigned char* hit, int grid) {
  emu_launch((unsigned)grid, pfc::kHnThreads, [=]() { pfc::similar_columns_kernel(a, n_a, b, n_b, emb, thr, hit); });
}
''',
    "bce_head": r'''
extern "C" void emu_bce_fwd(const float* feat, const float* weight, const float* bias, const int64_t* label, int64_t n_rows,
                            int64_t n_classes, int emb, float m, float r, float t, float* logits, unsigned char* gt,
                            float* cosine, float* inv_nf, float* inv_nw, int grid) {
  emu_launch((unsigned)grid, 256, [=]() {
    pfc::bce_head_fwd_kernel(feat, weight, bias, label, n_rows, n_classes, emb, m, r, t, logits, gt, cosine, inv_nf, inv_nw);
  });
}
extern "C" void emu_bce_bwd(const float* feat, const float* weight, const float* cosine, const float* inv_nf, const float* inv_nw,
                            const float* dlogits, int64_t n_rows, int64_t n_classes, int emb, float r, float t, float* dfeat,
                            float* dweight, float* dbias) {
  emu_launch((unsigned)(n_rows + n_classes), pfc::kBceThreads, [=]() {
    pfc::bce_head_bwd_kernel(feat, weight, cosine, inv_nf, inv_nw, dlogits, n_rows, n_classes, emb, r, t, dfeat, dweight, dbias);
  });
}
''',
}


# simt_check.cu's host functions are C++ (api.cu dispatches to them): export them for ctypes
CHECK_EXPORTS = r'''
extern "C" int emu_check_num_partials(int64_t n_rows, int64_t n_classes) { return pfc::simt_fwd_num_partials(n_rows, n_classes); }
extern "C" int emu_check_fwd_stats(const float* x, const float* w_hat, const int64_t* label, int64_t n_rows, int64_t n_classes, int emb,
                                   float s, float m, int kind, float* part_max, float* part_sum, float* target_logit) {
  return pfc::simt_fwd_stats(x, w_hat, label, n_rows, n_classes, emb, s, m, kind, part_max, part_sum, target_logit, nullptr);
}
extern "C" size_t emu_check_bwd_ws(int64_t n_rows, int64_t n_classes, int emb) { return pfc::simt_bwd_workspace_bytes(n_rows, n_classes, emb); }
extern "C" int emu_check_bwd(const float* x, const float* w_hat, const float* inv_norm, const int64_t* label, const float* row_max,
                             const float* row_sum, int64_t n_rows, int64_t n_classes, int emb, float s, float m, int kind, float inv_b,
                             float* dx, float* dw, int accumulate, void* ws, size_t ws_bytes) {
  return pfc::simt_bwd(x, w_hat, inv_norm, label, row_max, row_sum, n_rows, n_classes, emb, s, m, kind, inv_b, dx, dw, accumulate, ws, ws_bytes, nullptr);
}
'''


def _match_close(src, i, open_ch, close_ch):
    depth = 0
    for j in range(i, len(src)):
        if src[j] == open_ch:
            depth += 1
        elif src[j] == close_ch:
            depth -= 1
            if depth == 0:
                return j
    raise ValueError("unbalanced")


def _split_top(text):
    parts, depth, cur = [], 0, ""
    for ch in text:
        if ch in "([{":
            depth += 1
        elif ch in ")]}":
            depth -= 1
        if ch == "," and depth == 0:
            parts.append(cur)
            cur = ""
        else:
            cur += ch
    return parts + [cur]


def _transform_launches(src):
    """``kernel<T><<<grid, block, smem, stream>>>(args);`` -> ``emu_launch(grid, block, [=]() { kernel<T>(args); });``"""
    import re
    out, pos = "", 0
    while True:
        i = src.find("<<<", pos)
        if i < 0:
            return out + src[pos:]
        j = i                                           # walk back over the kernel name (+ template arguments)
        if src[j - 1] == ">":
            depth = 0
            while True:
                j -= 1
                depth += (src[j] == ">") - (src[j] == "<")
                if depth == 0:
                    break
        m = re.search(r"[\w:]+$", src[:j])
        name = src[m.start():i]
        k = src.index(">>>", i)
        cfg = _split_top(src[i + 3:k])
        a0 = src.index("(", k)
        a1 = _match_close(src, a0, "(", ")")
        out += src[pos:m.start()] + "emu_launch(EmuDim3(%s), (unsigned)(%s), [=]() { %s%s; })" % (
            cfg[0].strip(), cfg[1].strip(), name, src[a0:a1 + 1])
        pos = a1 + 1


def _build_abi(name, tmp, extra=""):
    """Whole translation unit (kernels AND the extern "C" entry points) on the emulator: launches become emu_launch,
    the CUDA runtime calls act on host memory."""
    src = open(os.path.join(ROOT, "fedfr_b200", "csrc", name + ".cu")).read() + extra
    for inc in ("rows_device.cuh",):                                  # in-tree device headers are inlined
        if '#include "%s"' % inc in src:
            src = src.replace('#include "%s"' % inc, open(os.path.join(ROOT, "fedfr_b200", "csrc", inc)).read())
    src = src.replace("#pragma once", "")
    body = _transform_launches(src.replace('#include "common.cuh"', '#include "cuda_emu.h"', 1).replace('#include "common.cuh"', ""))
    assert "<<<" not in body and "cuda_emu.h" in body
    cpp = os.path.join(tmp, name + "_abi_emu.cpp")
    with open(cpp, "w") as f:
        f.write(body)
    so = os.path.join(tmp, name + "_abi_emu.so")
    r = subprocess.run(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas"] + SAN_FLAGS +
                       ["-I", os.path.join(HERE, "emu"), cpp, "-o", so], capture_output=True, text=True)
    assert r.returncode == 0, "\n".join(l for l in r.stderr.splitlines() if "error" in l)[:1500]
    return C.CDLL(so)


def _build(name, tmp):
    src = open(os.path.join(ROOT, "fedfr_b200", "csrc", {"roc2": "roc"}.get(name, name) + ".cu")).read()
    end = src.index("}  // namespace pfc") + len("}  // namespace pfc")
    body = src[:end].replace('#include "common.cuh"', '#include "cuda_emu.h"')
    assert "cuda_emu.h" in body
    cpp = os.path.join(tmp, name + "_emu.cpp")
    with open(cpp, "w") as f:
        f.write(body + "\n" + HARNESS[name])
    so = os.path.join(tmp, name + "_emu.so")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas"] + SAN_FLAGS +
                          ["-I", os.path.join(HERE, "emu"), cpp, "-o", so])
    return C.CDLL(so)


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


@pytest.fixture(scope="module")
def libs(tmp_path_factory):
    import __graft_entry__ as g
    g.build()                                          # the C oracle
    tmp = str(tmp_path_factory.mktemp("emu"))
    out = {n: _build(n, tmp) for n in HARNESS}
    out.update({n + "_abi": _build_abi(n, tmp) for n in ("sample", "fedavg", "rows", "stats")})
    out["check_abi"] = _build_abi("simt_check", tmp, CHECK_EXPORTS)
    return out


@pytest.mark.parametrize("n,emb,t,off,grid", [(150, 40, 100, 0, 3), (131, 33, 131, 0, 2), (70, 7, 20, 35, 1), (64, 32, 64, 0, 5)])
def test_roc_kernel_under_emulation(libs, n, emb, t, off, grid):
    from oracle import roc_oracle as R
    rng = np.random.default_rng(n)
    f = rng.standard_normal((n, emb)).astype(np.float32)
    f /= np.linalg.norm(f, axis=1, keepdims=True)
    f[3] = f[1]
    f[n - 2] = -f[0]
    l = rng.integers(0, 5, n).astype(np.int32)
    sub, subl = np.ascontiguousarray(f[off:off + t]), np.ascontiguousarray(l[off:off + t])
    want = R.roc_histogram(f, l, sub, subl, off)
    hist = np.zeros(4002, dtype=np.uint64)
    libs["roc"].emu_roc(_p(f), _p(l), C.c_int64(n), _p(sub), _p(subl), C.c_int64(sub.shape[0]), C.c_int64(off), emb, _p(hist), grid)
    assert np.array_equal(hist.astype(np.int64), want)


@pytest.mark.parametrize("B,Cn,E,t,grid", [(9, 5, 40, 3, 2), (3, 300, 33, 2, 7), (20, 1, 130, 4, 1), (2, 2, 1024, 3, 1)])
def test_bce_head_kernels_under_emulation(libs, B, Cn, E, t, grid):
    from oracle import bce_head_oracle as O
    g = torch.Generator().manual_seed(B * 1000 + Cn)
    feat = (torch.randn(B, E, generator=g) * 2).numpy()
    weight = (torch.randn(Cn, E, generator=g) * 0.01).numpy()
    bias = (torch.randn(Cn, generator=g) * 0.1).numpy()
    label = torch.randint(-1, Cn + 3, (B,), generator=g).numpy()
    lo, gto, cso, nf, nw = O.forward(torch.from_numpy(feat).double(), torch.from_numpy(weight).double(),
                                     torch.from_numpy(bias).double(), torch.from_numpy(label), 0.4, 30.0, t)
    logits, gt = np.zeros((B, Cn), np.float32), np.zeros((B, Cn), np.uint8)
    cosine, inv_nf, inv_nw = np.zeros((B, Cn), np.float32), np.zeros(B, np.float32), np.zeros(Cn, np.float32)
    libs["bce_head"].emu_bce_fwd(_p(feat), _p(weight), _p(bias), _p(label), C.c_int64(B), C.c_int64(Cn), E, C.c_float(0.4),
                                 C.c_float(30.0), C.c_float(t), _p(logits), _p(gt), _p(cosine), _p(inv_nf), _p(inv_nw), grid)
    assert np.array_equal(gt.astype(bool), gto.numpy())
    np.testing.assert_allclose(logits, lo.numpy(), rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(cosine, cso.numpy(), rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(inv_nf, 1 / nf.numpy(), rtol=1e-5)
    np.testing.assert_allclose(inv_nw, 1 / nw.numpy(), rtol=1e-5)

    dlogits = torch.randn(B, Cn, generator=g).numpy()
    dfo, dwo, dbo = O.backward(torch.from_numpy(feat).double(), torch.from_numpy(weight).double(), cso, nf, nw,
                               torch.from_numpy(dlogits).double(), 30.0, t)
    dfeat, dweight, dbias = np.zeros_like(feat), np.zeros_like(weight), np.zeros_like(bias)
    libs["bce_head"].emu_bce_bwd(_p(feat), _p(weight), _p(cosine), _p(inv_nf), _p(inv_nw), _p(dlogits), C.c_int64(B),
                                 C.c_int64(Cn), E, C.c_float(30.0), C.c_float(t), _p(dfeat), _p(dweight), _p(dbias))
    for got, want in ((dfeat, dfo), (dweight, dwo), (dbias, dbo)):
        want = want.numpy()
        assert np.linalg.norm(got - want) <= 1e-5 * np.linalg.norm(want) + 1e-9

    # dfeat == NULL (detached features) and no bias: the class-role CTAs still produce dweight
    dweight2 = np.zeros_like(weight)
    libs["bce_head"].emu_bce_bwd(_p(feat), _p(weight), _p(cosine), _p(inv_nf), _p(inv_nw), _p(dlogits), C.c_int64(B),
                                 C.c_int64(Cn), E, C.c_float(30.0), C.c_float(t), None, _p(dweight2), None)
    assert np.array_equal(dweight2, dweight)


@pytest.mark.parametrize("na,nb,emb,thr,grid", [(70, 130, 40, 0.1, 3), (5, 64, 33, 0.0, 1), (130, 65, 7, 0.3, 4), (64, 64, 64, -2.0, 2)])
def test_similar_columns_kernel_under_emulation(libs, na, nb, emb, thr, grid):
    from oracle import hardneg_oracle as O
    rng = np.random.default_rng(na * 7 + nb)
    a = rng.standard_normal((na, emb)).astype(np.float32)
    a /= np.linalg.norm(a, axis=1, keepdims=True)
    b = (rng.standard_normal((nb, emb)) + 0.8 * a[rng.integers(0, na, nb)]).astype(np.float32)
    b /= np.linalg.norm(b, axis=1, keepdims=True)
    hit = np.zeros(nb, dtype=np.uint8)
    libs["hardneg"].emu_similar(_p(a), C.c_int64(na), _p(b), C.c_int64(nb), emb, C.c_float(thr), _p(hit), grid)
    certain, amb = O.similar_columns(a, b, thr)
    got = set(np.nonzero(hit)[0].tolist())
    assert set(certain.tolist()) <= got <= set(certain.tolist()) | set(amb.tolist())
    assert 0 < len(got) <= nb


# ------------------------------------------------------------------------------------------------------------------
# Whole C-ABI entry points under emulation (kernels + their host orchestration), against the REFERENCE goldens

def _sample_abi(lib, labels_global, perm, class_start, num_local, num_sample):
    """pfc_remap_labels + pfc_sample_index exactly as fedfr_b200.ops_cuda calls them; returns (index, remapped labels)."""
    lib.pfc_sample_workspace_bytes.restype = C.c_size_t
    n = labels_global.shape[0]
    local = np.empty(n, dtype=np.int64)
    assert lib.pfc_remap_labels(_p(labels_global), C.c_int64(n), C.c_int64(class_start), C.c_int64(num_local), _p(local), None) == 0
    perm = perm.astype(np.float32).copy()
    index = np.full(num_local, -7, dtype=np.int64)
    n_index = np.zeros(1, dtype=np.int64)
    ws_bytes = lib.pfc_sample_workspace_bytes(C.c_int64(num_local))
    ws = np.zeros(ws_bytes + 256, dtype=np.uint8)
    ws_ptr = (ws.ctypes.data + 255) // 256 * 256
    rc = lib.pfc_sample_index(_p(local), C.c_int64(n), _p(perm), C.c_int64(num_local), C.c_int64(num_sample), _p(index),
                              _p(n_index), C.c_void_p(ws_ptr), C.c_size_t(ws_bytes), None)
    assert rc == 0
    return index[:int(n_index[0])], local


@pytest.mark.parametrize("name", ["w1_sr01", "w1_sr_pos_overflow", "w2_sr03", "w2_arc_sr03"])
def test_sampling_abi_under_emulation_matches_reference(libs, name):
    """The sampled index the unmodified reference produced (partial_fc.py:89-106) must come out of the index kernel chain
    bit for bit, given the reference's own torch.rand draw."""
    sys.path.insert(0, HERE)
    from golden_util import Case
    from oracle import partial_fc_oracle as O
    case = Case(name)
    cfg = case.cfg
    W, C_all = cfg["world_size"], cfg["num_classes"]
    total = torch.cat(case.labels).numpy().astype(np.int64)
    for r in range(W):
        num_local = C_all // W + int(r < C_all % W)
        class_start = C_all // W * r + min(r, C_all % W)
        num_sample = int(cfg["sample_rate"] * num_local)
        for step in range(cfg["steps"]):
            if not case.has(r, step, "perm"):
                continue
            index, local = _sample_abi(libs["sample_abi"], total, case.get(r, step, "perm"), class_start, num_local, num_sample)
            assert np.array_equal(index, case.get(r, step, "index")), (name, r, step)
            want_local = O.relabel_to_sample(O.remap_labels(total, class_start, num_local), case.get(r, step, "index"))
            assert np.array_equal(local, want_local)


@pytest.mark.parametrize("num_local,n_label,num_sample,seed", [(5000, 64, 500, 0), (2049, 300, 100, 1), (300, 10, 0, 2), (257, 4, 257, 3)])
def test_sampling_abi_under_emulation_matches_oracle(libs, num_local, n_label, num_sample, seed):
    from oracle import partial_fc_oracle as O
    rng = np.random.default_rng(seed)
    perm = rng.random(num_local, dtype=np.float32)
    perm[rng.integers(0, num_local, 6)] = perm[0]                       # ties, also at the threshold for some k
    labels = rng.integers(-50, num_local + 50, n_label).astype(np.int64)
    index, local = _sample_abi(libs["sample_abi"], labels, perm, 0, num_local, num_sample)
    local0 = O.remap_labels(labels, 0, num_local)
    want = O.sample_index(local0, perm, num_sample)
    assert np.array_equal(index, want)
    assert np.array_equal(local, O.relabel_to_sample(local0, want))


def test_fedavg_abi_under_emulation_matches_reference(libs):
    """fedavg_weighted_sum (pointer table, fp32 + int64 segments, ragged tails) and fedavg_blend against the outputs of the
    unmodified server.FedPavg / FedAvg_on_FC (tests/golden/fedavg.npz) -- bit for bit."""
    from oracle import partial_fc_oracle as O
    lib = libs["fedavg_abi"]
    lib.fedavg_table_bytes.restype = C.c_size_t
    z = np.load(os.path.join(HERE, "golden", "fedavg.npz"))
    K = int(z["K"])
    keys = [k[4:] for k in z.files if k.startswith("in0/")]
    wn = np.array([np.float32(w) for w in O.fedavg_weights([float(w) for w in z["weights"]])], dtype=np.float32)
    srcs = [[np.ascontiguousarray(z[f"in{i}/{k}"]) for i in range(K)] for k in keys]
    outs = [np.full(max(g[0].size, 1), np.nan, dtype=np.float32) for g in srcs]
    n_seg = len(keys)
    seg_src = np.array([a.ctypes.data for g in srcs for a in g], dtype=np.uint64)
    seg_out = np.array([o.ctypes.data for o in outs], dtype=np.uint64)
    seg_len = np.array([g[0].size for g in srcs], dtype=np.int64)
    seg_dtype = np.array([1 if g[0].dtype == np.int64 else 0 for g in srcs], dtype=np.int32)
    assert all(g[0].dtype in (np.float32, np.int64) for g in srcs) and seg_dtype.sum() >= 1
    tb = lib.fedavg_table_bytes(n_seg, K)
    table = np.zeros(tb + 256, dtype=np.uint8)
    rc = lib.fedavg_weighted_sum(_p(seg_src), _p(seg_out), _p(seg_len), _p(seg_dtype), n_seg, _p(wn), K,
                                 C.c_void_p((table.ctypes.data + 255) // 256 * 256), C.c_size_t(tb), None)
    assert rc == 0
    for k, o, g in zip(keys, outs, srcs):
        want = np.asarray(z["out/" + k], dtype=np.float32).reshape(-1)
        assert np.array_equal(o[:want.size], want), k

    fcs = [np.ascontiguousarray(z[f"fc_in{i}"]) for i in range(K)]
    aggr = np.empty_like(fcs[0])
    seg_src = np.array([a.ctypes.data for a in fcs], dtype=np.uint64)
    seg_out = np.array([aggr.ctypes.data], dtype=np.uint64)
    rc = lib.fedavg_weighted_sum(_p(seg_src), _p(seg_out), _p(np.array([aggr.size], dtype=np.int64)), _p(np.zeros(1, np.int32)), 1,
                                 _p(wn), K, C.c_void_p((table.ctypes.data + 255) // 256 * 256), C.c_size_t(tb), None)
    assert rc == 0 and np.array_equal(aggr, z["fc_out_p1"])
    out = np.empty_like(aggr)
    old = np.ascontiguousarray(z["fc_old"])
    assert lib.fedavg_blend(_p(old), _p(aggr), C.c_float(np.float32(1 - 0.7)), C.c_float(np.float32(0.7)), C.c_int64(aggr.size), _p(out), None) == 0
    assert np.array_equal(out, z["fc_out_p07"])


def _bf16_bits(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(torch.bfloat16).view(torch.int16).numpy()


@pytest.mark.parametrize("n_src,emb,gather", [(37, 512, False), (50, 128, True), (9, 64, True), (5, 1024, False)])
def test_row_kernels_abi_under_emulation(libs, n_src, emb, gather):
    """normalize (+gather) / cast / gather / scatter (partial_fc.py:105-106,113-116,127) through their C-ABI entries."""
    import torch.nn.functional as F
    lib = libs["rows_abi"]
    rng = np.random.default_rng(n_src + emb)
    w = (rng.standard_normal((n_src, emb)) * 0.01).astype(np.float32)
    w[1] = 0.0                                                            # the eps clamp of F.normalize
    mom = (rng.standard_normal((n_src, emb)) * 0.001).astype(np.float32)
    index = np.sort(rng.choice(n_src, size=n_src // 2, replace=False)).astype(np.int64) if gather else None
    rows = w[index] if gather else w
    n = rows.shape[0]
    w_bf16 = np.zeros((n, emb), dtype=np.int16)
    w_f32 = np.zeros((n, emb), dtype=np.float32)
    inv = np.zeros(n, dtype=np.float32)
    assert lib.pfc_normalize_rows(_p(w), _p(index), C.c_int64(n), emb, _p(w_bf16), _p(w_f32), _p(inv), None) == 0
    want = F.normalize(torch.from_numpy(rows)).numpy()
    np.testing.assert_allclose(w_f32, want, rtol=4e-7, atol=0)           # a division by the norm; the norm's summation
                                                                         # order differs from CPU torch's by <= 1 ulp
    np.testing.assert_allclose(inv, 1.0 / np.maximum(np.linalg.norm(rows.astype(np.float64), axis=1), 1e-12), rtol=2e-6)
    assert np.array_equal(w_bf16, _bf16_bits(w_f32))                     # the bf16 copy is the rounding of the fp32 one
    bf_only = np.zeros((n, emb), dtype=np.int16)                          # product mode: bf16 only (reciprocal multiply)
    assert lib.pfc_normalize_rows(_p(w), _p(index), C.c_int64(n), emb, _p(bf_only), None, _p(inv), None) == 0
    assert np.abs(bf_only.astype(np.int32) - _bf16_bits(want).astype(np.int32)).max() <= 1

    cast = np.zeros((n_src, emb), dtype=np.int16)
    assert lib.pfc_cast_rows_bf16(_p(w), C.c_int64(n_src), emb, _p(cast), None) == 0
    assert np.array_equal(cast, _bf16_bits(w))

    if gather:
        sub_w, sub_m = np.zeros((n, emb), np.float32), np.zeros((n, emb), np.float32)
        assert lib.pfc_gather_rows2(_p(w), _p(mom), _p(index), C.c_int64(n), emb, _p(sub_w), _p(sub_m), None) == 0
        assert np.array_equal(sub_w, w[index]) and np.array_equal(sub_m, mom[index])
        w2, m2 = w.copy(), mom.copy()
        new_w, new_m = sub_w + 1.0, sub_m - 1.0
        assert lib.pfc_scatter_rows2(_p(w2), _p(m2), _p(index), C.c_int64(n), emb, _p(new_w), _p(new_m), None) == 0
        ew, em = w.copy(), mom.copy()
        ew[index], em[index] = new_w, new_m
        assert np.array_equal(w2, ew) and np.array_equal(m2, em)


@pytest.mark.parametrize("sampled,nesterov,dampening,wd", [(False, 0, 0.0, 5e-4), (True, 0, 0.0, 5e-4), (False, 1, 0.0, 0.0), (True, 0, 0.1, 1e-3)])
def test_sgd_step_abi_under_emulation_matches_torch(libs, sampled, nesterov, dampening, wd):
    """pfc_sgd_step == torch.optim.SGD.step() (+ update() when sampled) on the same numbers, two consecutive steps."""
    lib = libs["rows_abi"]
    g = torch.Generator().manual_seed(11 + nesterov)
    n_all, emb = 40, 128
    weight = torch.randn(n_all, emb, generator=g) * 0.01
    mom = torch.randn(n_all, emb, generator=g) * 0.001
    index = torch.sort(torch.randperm(n_all, generator=g)[:17])[0] if sampled else None
    w_np, m_np = weight.numpy().copy(), mom.numpy().copy()
    for step in range(2):
        n = 17 if sampled else n_all
        grad = torch.randn(n, emb, generator=g) * 0.1
        sub = torch.nn.Parameter((weight[index] if sampled else weight).clone())
        sub.grad = grad.clone()
        opt = torch.optim.SGD([sub], lr=0.1, momentum=0.9, dampening=dampening, weight_decay=wd, nesterov=bool(nesterov))
        opt.state[sub]["momentum_buffer"] = (mom[index] if sampled else mom).clone()      # partial_fc.py:126
        opt.step()
        if sampled:                                                                        # partial_fc.py:113-116
            mom[index] = opt.state[sub]["momentum_buffer"]
            weight[index] = sub.data
        else:
            weight, mom = sub.data.clone(), opt.state[sub]["momentum_buffer"].clone()
        w_hat = np.zeros((n_all, emb), np.int16)
        inv = np.zeros(n_all, np.float32)
        rc = lib.pfc_sgd_step(_p(w_np), _p(m_np), _p(grad.numpy()), _p(index.numpy()) if sampled else None, C.c_int64(n), emb,
                              C.c_float(0.1), C.c_float(0.9), C.c_float(dampening), C.c_float(wd), nesterov,
                              None if sampled else _p(w_hat), None if sampled else _p(inv), None)
        assert rc == 0
        np.testing.assert_allclose(w_np, weight.numpy(), rtol=0, atol=2e-9)
        np.testing.assert_allclose(m_np, mom.numpy(), rtol=0, atol=2e-8)
        if not sampled:                                                   # the operands of the next forward
            want = torch.nn.functional.normalize(torch.from_numpy(w_np)).numpy()
            assert np.abs(w_hat.astype(np.int32) - _bf16_bits(want).astype(np.int32)).max() <= 1
            np.testing.assert_allclose(inv, 1.0 / np.linalg.norm(w_np.astype(np.float64), axis=1), rtol=2e-6)


def test_cosface_dense_abi_under_emulation(libs):
    """losses.CosFace.forward on materialised logits (losses.py:23-29): in-place margin, then a scaled copy."""
    lib = libs["rows_abi"]
    g = torch.Generator().manual_seed(3)
    cosine = torch.rand(19, 41, generator=g) * 2 - 1
    label = torch.randint(0, 41, (19,), generator=g)
    label[::4] = -1
    want_c = cosine.clone()
    rows = torch.where(label != -1)[0]
    want_c[rows, label[rows]] -= 0.4
    c_np, out = cosine.numpy().copy(), np.zeros((19, 41), np.float32)
    assert lib.pfc_cosface_dense(_p(c_np), _p(label.numpy()), C.c_int64(19), C.c_int64(41), C.c_float(64.0), C.c_float(0.4), _p(out), None) == 0
    assert np.array_equal(c_np, want_c.numpy()) and np.array_equal(out, (want_c * 64.0).numpy())


def test_arcface_dense_abi_under_emulation(libs):
    """losses.ArcFace.forward on materialised logits (losses.py:38-45): acos_ over the matrix, + m on the target column of
    the rows with a label, cos_, mul_(s) -- in place, one pass."""
    lib = libs["rows_abi"]
    g = torch.Generator().manual_seed(4)
    cosine = torch.rand(23, 37, generator=g) * 1.998 - 0.999
    cosine[0, 0], cosine[1, 1] = 1.0, -1.0                      # the ends of acos
    label = torch.randint(0, 37, (23,), generator=g)
    label[::5] = -1
    label[0], label[1] = 0, 1
    want = cosine.clone()
    rows = torch.where(label != -1)[0]
    want.acos_()
    want[rows, label[rows]] += 0.5
    want.cos_().mul_(64.0)
    c_np = cosine.numpy().copy()
    assert lib.pfc_arcface_dense(_p(c_np), _p(label.numpy()), C.c_int64(23), C.c_int64(37), C.c_float(64.0), C.c_float(0.5), None) == 0
    np.testing.assert_allclose(c_np, want.numpy(), rtol=0, atol=64.0 * 4e-7)
    assert lib.pfc_arcface_dense(_p(c_np), _p(label.numpy()), C.c_int64(0), C.c_int64(37), C.c_float(64.0), C.c_float(0.5), None) == 0


@pytest.mark.parametrize("world,n_rows,n_part", [(1, 33, 5), (3, 70, 2), (2, 1100, 1)])
def test_stats_abi_under_emulation(libs, world, n_rows, n_part):
    """pfc_merge_stats + pfc_finalize_stats == the reference's max / sum-exp / target all-reduces and loss
    (partial_fc.py:140-162), from per-tile partials."""
    lib = libs["stats_abi"]
    rng = np.random.default_rng(world * 100 + n_rows)
    C_per = 24
    z = (rng.standard_normal((world, n_part, n_rows, C_per)) * 20).astype(np.float32)      # logits per rank / partial slot
    owner = rng.integers(0, world, n_rows)
    tcol = rng.integers(0, n_part * C_per, n_rows)
    gathered = np.zeros((world, n_rows, 3), np.float32)
    for r in range(world):
        pm = z[r].max(axis=2)                                                               # [n_part, n_rows]
        ps = np.exp(z[r] - pm[:, :, None]).sum(axis=2).astype(np.float32)
        tl = np.zeros(n_rows, np.float32)
        mine = owner == r
        flat = z[r].transpose(1, 0, 2).reshape(n_rows, -1)
        tl[mine] = flat[mine, tcol[mine]]
        stats = np.zeros((n_rows, 3), np.float32)
        assert lib.pfc_merge_stats(_p(np.ascontiguousarray(pm)), _p(np.ascontiguousarray(ps)), _p(tl), n_part, C.c_int64(n_rows), _p(stats), None) == 0
        gathered[r] = stats
    row_max, row_sum, loss = np.zeros(n_rows, np.float32), np.zeros(n_rows, np.float32), np.zeros(1, np.float32)
    assert lib.pfc_finalize_stats(_p(gathered), world, C.c_int64(n_rows), _p(row_max), _p(row_sum), _p(loss), None) == 0
    full = z.transpose(2, 0, 1, 3).reshape(n_rows, -1).astype(np.float64)
    M = full.max(axis=1)
    S = np.exp(full - M[:, None]).sum(axis=1)
    tz = np.array([z[owner[i]].transpose(1, 0, 2).reshape(n_rows, -1)[i, tcol[i]] for i in range(n_rows)], dtype=np.float64)
    want_loss = -np.mean(np.log(np.maximum(np.exp(tz - M) / S, 1e-30)))
    np.testing.assert_allclose(row_max, M, rtol=1e-6)
    np.testing.assert_allclose(row_sum, S, rtol=1e-5)
    assert abs(float(loss[0]) - want_loss) < 1e-5 * abs(want_loss)


@pytest.mark.parametrize("name", ["w1_sr1_small", "w1_sr1_s30", "w1_arc_small", "w2_sr1_ragged"])
def test_check_mode_path_under_emulation_matches_reference(libs, name):
    """The fp32 check-mode kernels (PFC_PATH_CHECK: simt_check.cu + rows.cu + stats.cu), chained exactly as
    fedfr_b200.PartialFC.forward_backward chains them, against loss / x_grad / dw of the unmodified reference
    (partial_fc.py:130-176) -- tolerance 1e-4 relative, the north-star check-mode bar."""
    sys.path.insert(0, HERE)
    from golden_util import Case
    case = Case(name)
    cfg = case.cfg
    W, B, E = cfg["world_size"], cfg["batch"], cfg["emb"]
    kind = 1 if cfg.get("loss", "cosface") == "arcface" else 0
    s_, m_ = float(cfg["s"]), float(cfg["m"])
    rows_lib, stats_lib, chk, smp = libs["rows_abi"], libs["stats_abi"], libs["check_abi"], libs["sample_abi"]
    chk.emu_check_bwd_ws.restype = C.c_size_t
    x = np.ascontiguousarray(torch.cat(case.features).numpy())                       # the all-gathered batch
    total_label = torch.cat(case.labels).numpy().astype(np.int64)
    Bt = B * W
    per_rank, gathered = [], np.zeros((W, Bt, 3), np.float32)
    for r in range(W):
        w = np.ascontiguousarray(case.weights[r].numpy())
        Cl = w.shape[0]
        class_start = cfg["num_classes"] // W * r + min(r, cfg["num_classes"] % W)
        local = np.empty(Bt, np.int64)
        assert smp.pfc_remap_labels(_p(total_label), C.c_int64(Bt), C.c_int64(class_start), C.c_int64(Cl), _p(local), None) == 0
        w_hat, inv = np.zeros((Cl, E), np.float32), np.zeros(Cl, np.float32)
        assert rows_lib.pfc_normalize_rows(_p(w), None, C.c_int64(Cl), E, None, _p(w_hat), _p(inv), None) == 0
        n_part = chk.emu_check_num_partials(C.c_int64(Bt), C.c_int64(Cl))
        pm, ps, tl = np.zeros((n_part, Bt), np.float32), np.zeros((n_part, Bt), np.float32), np.zeros(Bt, np.float32)
        assert chk.emu_check_fwd_stats(_p(x), _p(w_hat), _p(local), C.c_int64(Bt), C.c_int64(Cl), E, C.c_float(s_), C.c_float(m_), kind,
                                       _p(pm), _p(ps), _p(tl)) == 0
        stats = np.zeros((Bt, 3), np.float32)
        assert stats_lib.pfc_merge_stats(_p(pm), _p(ps), _p(tl), n_part, C.c_int64(Bt), _p(stats), None) == 0
        gathered[r] = stats                                                          # the one all-gather of the W > 1 path
        per_rank.append((w_hat, inv, local, Cl))
    row_max, row_sum, loss = np.zeros(Bt, np.float32), np.zeros(Bt, np.float32), np.zeros(1, np.float32)
    assert stats_lib.pfc_finalize_stats(_p(gathered), W, C.c_int64(Bt), _p(row_max), _p(row_sum), _p(loss), None) == 0
    dx_sum = np.zeros((Bt, E), np.float64)
    for r, (w_hat, inv, local, Cl) in enumerate(per_rank):
        ws_bytes = chk.emu_check_bwd_ws(C.c_int64(Bt), C.c_int64(Cl), E)
        ws = np.zeros(ws_bytes // 4 + 64, np.float32)
        dx, dw = np.zeros((Bt, E), np.float32), np.zeros((Cl, E), np.float32)
        assert chk.emu_check_bwd(_p(x), _p(w_hat), _p(inv), _p(local), _p(row_max), _p(row_sum), C.c_int64(Bt), C.c_int64(Cl), E,
                                 C.c_float(s_), C.c_float(m_), kind, C.c_float(1.0 / Bt), _p(dx), _p(dw), 0, _p(ws), C.c_size_t(ws_bytes)) == 0
        dx_sum += dx
        want_dw = case.get(r, 0, "dw")
        assert np.linalg.norm(dw - want_dw) < 1e-4 * np.linalg.norm(want_dw), (name, r)
    for r in range(W):                                                               # reduce-scatter + x W (partial_fc.py:171-174)
        assert abs(float(loss[0]) - float(case.get(r, 0, "loss"))) < 1e-4 * abs(float(case.get(r, 0, "loss")))
        got = dx_sum[r * B:(r + 1) * B] * W
        want = case.get(r, 0, "x_grad")
        assert np.linalg.norm(got - want) < 1e-4 * np.linalg.norm(want), (name, r)


def test_new_entry_points_with_the_product_ctypes_signatures(libs, tmp_path):
    """pfc_bce_head_fwd/bwd, pfc_similar_columns and pfc_roc_histogram called on the emulated build with the argtypes of
    fedfr_b200/_native.py and arguments marshalled the way the Python wrappers marshal them (data_ptr ints, Python
    ints/floats, None for NULL): catches a signature drift between include/fedfr_b200.h, the .cu files and _native.py."""
    from fedfr_b200 import _native as N
    from oracle import bce_head_oracle as OB, hardneg_oracle as OH, roc_oracle as OR
    built = {"pfc_bce_head_fwd": _build_abi("bce_head", str(tmp_path)), "pfc_similar_columns": _build_abi("hardneg", str(tmp_path)),
             "pfc_roc_histogram": _build_abi("roc", str(tmp_path))}
    built["pfc_bce_head_bwd"] = built["pfc_bce_head_fwd"]
    fn = {}
    for name, lib in built.items():
        f = getattr(lib, name)
        f.restype, f.argtypes = N.SIGNATURES[name]
        fn[name] = f
    g = torch.Generator().manual_seed(5)
    B, Cn, E = 6, 4, 48
    feat, weight, bias = torch.randn(B, E, generator=g), torch.randn(Cn, E, generator=g) * 0.01, torch.randn(Cn, generator=g)
    y = torch.tensor([0, 3, 9, 1, 2, 2])
    logits, gt, cosine = torch.empty(B, Cn), torch.empty(B, Cn, dtype=torch.uint8), torch.empty(B, Cn)
    inv_nf, inv_nw = torch.empty(B), torch.empty(Cn)
    assert fn["pfc_bce_head_fwd"](N.ptr(feat), N.ptr(weight), N.ptr(bias), N.ptr(y), B, Cn, E, 0.4, 30.0, 3.0, N.ptr(logits), N.ptr(gt),
                                  N.ptr(cosine), N.ptr(inv_nf), N.ptr(inv_nw), None) == 0
    lo, gto, cso, nf, nw = OB.forward(feat.double(), weight.double(), bias.double(), y, 0.4, 30.0, 3)
    assert torch.equal(gt.bool(), gto) and torch.allclose(logits.double(), lo, rtol=1e-5, atol=1e-5)
    dlogits = torch.randn(B, Cn, generator=g)
    dfeat, dweight, dbias = torch.empty(B, E), torch.empty(Cn, E), torch.empty(Cn)
    assert fn["pfc_bce_head_bwd"](N.ptr(feat), N.ptr(weight), N.ptr(cosine), N.ptr(inv_nf), N.ptr(inv_nw), N.ptr(dlogits), B, Cn, E, 30.0, 3.0,
                                  N.ptr(dfeat), N.ptr(dweight), N.ptr(dbias), None) == 0
    dfo, dwo, dbo = OB.backward(feat.double(), weight.double(), cso, nf, nw, dlogits.double(), 30.0, 3)
    assert torch.allclose(dfeat.double(), dfo, rtol=1e-4, atol=1e-7) and torch.allclose(dweight.double(), dwo, rtol=1e-4, atol=1e-6)
    assert torch.allclose(dbias.double(), dbo, rtol=1e-5, atol=1e-6)

    a = torch.nn.functional.normalize(torch.randn(10, E, generator=g))
    b = torch.nn.functional.normalize(torch.randn(70, E, generator=g))
    hit = torch.full((70,), 7, dtype=torch.uint8)
    assert fn["pfc_similar_columns"](N.ptr(a), a.shape[0], N.ptr(b), b.shape[0], E, 0.2, N.ptr(hit), None) == 0
    certain, amb = OH.similar_columns(a.numpy(), b.numpy(), 0.2)
    got = set(torch.nonzero(hit, as_tuple=True)[0].tolist())
    assert set(certain.tolist()) <= got <= set(certain.tolist()) | set(amb.tolist()) and int(hit.max()) <= 1

    lab = torch.randint(0, 3, (70,), generator=g).int()
    out = torch.zeros(4002, dtype=torch.int64)
    assert fn["pfc_roc_histogram"](N.ptr(b), N.ptr(lab), 70, N.ptr(b[20:50]), N.ptr(lab[20:50]), 30, 20, E, N.ptr(out), None) == 0
    assert np.array_equal(out.numpy(), OR.roc_histogram(b.numpy(), lab.numpy(), b[20:50].numpy(), lab[20:50].numpy(), 20))


@pytest.mark.parametrize("kind,n,emb,t,off,grid", [("random", 150, 40, 100, 0, 3), ("random", 70, 512, 40, 0, 2), ("edges", 96, 64, 96, 0, 2),
                                                  ("edges", 70, 33, 30, 20, 1), ("scaled", 80, 100, 80, 0, 4),
                                                  ("alledges", 128, 16, 128, 0, 1), ("halfedges", 200, 24, 150, 0, 2)])
def test_two_tier_roc_kernel_is_integer_identical(libs, kind, n, emb, t, off, grid):
    """roc_hist2_kernel (fp32 FMA filter + exact chain near bin edges) must reproduce the exact kernel's histogram for every
    input -- including rows whose cosine sits EXACTLY on a bin edge (one-hot, duplicate, opposite, zero rows)."""
    from oracle import roc_oracle as R
    rng = np.random.default_rng(n + emb)
    f = rng.standard_normal((n, emb)).astype(np.float32)
    f /= np.linalg.norm(f, axis=1, keepdims=True)
    if kind == "edges":
        for r in range(0, n, 3):                       # one-hot rows: dots are exactly 0 or 1 -> x = 1000 / 2000 on the edge
            f[r] = 0
            f[r, (r // 3) % emb] = 1.0
        f[1] = f[4]
        f[7] = -f[4]
        f[10] = 0.0
        f[13] = 0.5 * f[16]                            # cosine-like value 0.5 * |f16|^2 ~ 0.5 -> x ~ 1500 (edge or a hair off it)
    if kind == "scaled":
        f *= rng.uniform(0.2, 1.0, (n, 1)).astype(np.float32)
    if kind in ("alledges", "halfedges"):              # every (or every other) pair on a bin edge: the exact-chain queue of a CTA
        for r in range(0, n, 1 if kind == "alledges" else 2):          # overflows / is drained several times across tiles
            f[r] = 0
            f[r, r % emb] = 1.0
    l = rng.integers(0, 5, n).astype(np.int32)
    sub, subl = np.ascontiguousarray(f[off:off + t]), np.ascontiguousarray(l[off:off + t])
    want = R.roc_histogram(f, l, sub, subl, off)
    coef = np.float32((32 + (emb + 31) // 32 + 2) * 2.0 ** -24)
    hist = np.zeros(4002, dtype=np.uint64)
    libs["roc2"].emu_roc2(_p(f), _p(l), C.c_int64(n), _p(sub), _p(subl), C.c_int64(sub.shape[0]), C.c_int64(off), emb, C.c_float(coef),
                          _p(hist), grid)
    assert np.array_equal(hist.astype(np.int64), want)
    exact = np.zeros(4002, dtype=np.uint64)
    libs["roc"].emu_roc(_p(f), _p(l), C.c_int64(n), _p(sub), _p(subl), C.c_int64(sub.shape[0]), C.c_int64(off), emb, _p(exact), grid)
    assert np.array_equal(hist, exact)


@pytest.mark.skipif(os.environ.get("EMU_ASAN") == "1", reason="this IS the sanitizer child")
def test_emulated_kernels_under_address_sanitizer():
    """memcheck on the CPU: every test of this file again in a child process whose emulated builds are compiled with
    -fsanitize=address (shared-memory arrays are instrumented globals, "device" buffers are malloc'd numpy arrays with red
    zones), so an out-of-bounds load or store in any emulated kernel aborts the child.  The child also runs threads and
    blocks in DESCENDING order (EMU_SCHEDULE=reverse): results that depend on a missing barrier differ between the two orders."""
    asan = subprocess.run(["gcc", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(asan) or not os.path.exists(asan):
        pytest.skip("libasan not available")
    env = dict(os.environ, LD_PRELOAD=asan, EMU_ASAN="1", EMU_SCHEDULE="reverse",      # and the opposite thread/block order
               ASAN_OPTIONS="detect_leaks=0:detect_stack_use_after_return=0",
               CUDA_VISIBLE_DEVICES="")      # the emulation needs no device: keep the GPU driver out of the instrumented process
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-p", "no:cacheprovider",
                        "-k", "not property and not sgd_step and not stats_abi and not check_mode"],     # time budget: the sweeps and
                       # the slowest B200-validated kernels stay in the plain pass only
                       env=env, capture_output=True, text=True, cwd=ROOT, timeout=1500)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0 and "AddressSanitizer" not in r.stdout + r.stderr.replace(
        "ASan doesn't fully support makecontext/swapcontext", ""), tail


def test_c_abi_error_codes_under_emulation(libs, tmp_path):
    """The argument checks of the C ABI (include/fedfr_b200.h: 0 ok, PFC_E_ARG -1, PFC_E_SHAPE -2, PFC_E_WORKSPACE -4) return
    before any launch -- exercised here on the emulated builds, where require_sm100() passes without a GPU."""
    E_ARG, E_SHAPE, E_WS = -1, -2, -4
    smp, rows = libs["sample_abi"], libs["rows_abi"]
    smp.pfc_sample_workspace_bytes.restype = C.c_size_t
    lab, perm, idx = np.zeros(4, np.int64), np.zeros(16, np.float32), np.zeros(16, np.int64)
    ws = np.zeros(smp.pfc_sample_workspace_bytes(C.c_int64(16)) + 256, np.uint8)
    wsp, wsb = C.c_void_p((ws.ctypes.data + 255) // 256 * 256), C.c_size_t(ws.size - 256)

    def sample(label=lab, n_label=4, p=perm, num_local=16, num_sample=4, index=idx, w=wsp, wb=wsb):
        return smp.pfc_sample_index(_p(label), C.c_int64(n_label), _p(p), C.c_int64(num_local), C.c_int64(num_sample), _p(index), None, w, wb, None)
    assert sample() == 0
    assert sample(label=None) == E_ARG and sample(num_local=0) == E_ARG and sample(num_sample=-1) == E_ARG
    assert sample(num_sample=17) == E_SHAPE                       # more samples than local classes
    assert sample(wb=C.c_size_t(8)) == E_WS
    assert smp.pfc_remap_labels(None, C.c_int64(4), C.c_int64(0), C.c_int64(4), _p(lab), None) == E_ARG
    assert smp.pfc_remap_labels(_p(lab), C.c_int64(0), C.c_int64(0), C.c_int64(4), _p(lab), None) == 0       # empty batch

    x = np.zeros((2, 6), np.float32)
    out = np.zeros((2, 6), np.int16)
    assert rows.pfc_cast_rows_bf16(_p(x), C.c_int64(2), 6, _p(out), None) == E_ARG                            # emb % 4 != 0
    assert rows.pfc_cast_rows_bf16(_p(x), C.c_int64(0), 8, _p(out), None) == 0

    bce = _build_abi("bce_head", str(tmp_path))
    f = np.zeros((2, 8), np.float32)
    assert bce.pfc_bce_head_bwd(_p(f), _p(f), _p(f), _p(f), _p(f), _p(f), C.c_int64(2), C.c_int64(2), 2048, C.c_float(30), C.c_float(3),
                                _p(f), _p(f), None, None) == E_SHAPE                                          # emb > 1024
    assert bce.pfc_bce_head_fwd(None, _p(f), None, _p(lab), C.c_int64(2), C.c_int64(2), 8, C.c_float(.4), C.c_float(30), C.c_float(3),
                                _p(f), _p(f), _p(f), _p(f), _p(f), None) == E_ARG
    roc = _build_abi("roc", str(tmp_path))
    l32 = np.zeros(2, np.int32)
    assert roc.pfc_roc_histogram(_p(f), _p(l32), C.c_int64(2), _p(f), _p(l32), C.c_int64(2), C.c_int64(0), 8, None, None) == E_ARG
    assert roc.pfc_roc_histogram(_p(f), _p(l32), C.c_int64(2), _p(f), _p(l32), C.c_int64(2), C.c_int64(-1), 8, _p(np.zeros(4002, np.int64)), None) == E_ARG
    assert roc.pfc_set_roc_mode(2) == E_ARG and roc.pfc_set_roc_mode(0) == 0
    hn = _build_abi("hardneg", str(tmp_path))
    hit = np.zeros(2, np.uint8)
    assert hn.pfc_similar_columns(_p(f), C.c_int64(2), _p(f), C.c_int64(2), 0, C.c_float(.2), _p(hit), None) == E_ARG
    assert hn.pfc_similar_columns(_p(f), C.c_int64(2), _p(f), C.c_int64(2), 8, C.c_float(.2), None, None) == E_ARG


def test_sampling_abi_under_emulation_property(libs):
    """Random shard sizes, label batches (incl. none owned, all owned, duplicates) and perm draws quantised to force ties
    at the k-th value: the index kernel chain equals the oracle's topk + sort + searchsorted every time."""
    from hypothesis import given, settings, strategies as st
    from oracle import partial_fc_oracle as O

    @settings(max_examples=30, deadline=None, derandomize=True)
    @given(st.integers(1, 2600), st.integers(0, 150), st.floats(0.0, 1.0), st.integers(0, 2 ** 31 - 1), st.sampled_from([0, 4, 64, 4096]))
    def run(num_local, n_label, rate, seed, quant):
        rng = np.random.default_rng(seed)
        perm = rng.random(num_local, dtype=np.float32)
        if quant:
            perm = (np.floor(perm * quant) / quant).astype(np.float32)      # heavy ties
        labels = rng.integers(-20, num_local + 20, n_label).astype(np.int64)
        num_sample = int(rate * num_local)
        index, local = _sample_abi(libs["sample_abi"], labels, perm, 0, num_local, num_sample)
        local0 = O.remap_labels(labels, 0, num_local)
        want = O.sample_index(local0, perm, num_sample)
        assert np.array_equal(index, want)
        assert np.array_equal(local, O.relabel_to_sample(local0, want))
    run()


def test_fedavg_abi_under_emulation_property(libs):
    """Random client counts, segment counts and lengths around the vector / block boundaries (0, 1, 3, 4, 5, 1023, 1024,
    1025 ...), fp32 and int64 segments: fedavg_weighted_sum equals the sequential fp32 multiply-then-add of server.py:30-33
    bit for bit."""
    from hypothesis import given, settings, strategies as st
    from oracle import partial_fc_oracle as O
    lib = libs["fedavg_abi"]
    lib.fedavg_table_bytes.restype = C.c_size_t
    lens = st.sampled_from([0, 1, 3, 4, 5, 7, 8, 255, 1023, 1024, 1025, 2048, 3001])

    @settings(max_examples=25, deadline=None, derandomize=True)
    @given(st.integers(1, 9), st.lists(st.tuples(lens, st.booleans()), min_size=1, max_size=5), st.integers(0, 2 ** 31 - 1))
    def run(K, segs, seed):
        rng = np.random.default_rng(seed)
        weights = [float(w) for w in rng.integers(1, 10000, K)]
        wn = np.array([np.float32(w) for w in O.fedavg_weights(weights)], dtype=np.float32)
        models = []
        for i in range(K):
            sd = {}
            for s, (n, is_int) in enumerate(segs):
                sd[f"t{s}"] = rng.integers(0, 100000, n).astype(np.int64) if is_int else rng.standard_normal(n).astype(np.float32)
            models.append(sd)
        keys = list(models[0].keys())
        srcs = [[np.ascontiguousarray(m[k]) for m in models] for k in keys]
        outs = [np.full(max(g[0].size, 4), np.nan, dtype=np.float32) for g in srcs]
        assert all(a.ctypes.data % 16 == 0 or a.size < 4 for g in srcs for a in g)
        seg_src = np.array([a.ctypes.data for g in srcs for a in g], dtype=np.uint64)
        seg_out = np.array([o.ctypes.data for o in outs], dtype=np.uint64)
        seg_len = np.array([g[0].size for g in srcs], dtype=np.int64)
        seg_dtype = np.array([1 if g[0].dtype == np.int64 else 0 for g in srcs], dtype=np.int32)
        tb = lib.fedavg_table_bytes(len(keys), K)
        table = np.zeros(tb + 256, dtype=np.uint8)
        rc = lib.fedavg_weighted_sum(_p(seg_src), _p(seg_out), _p(seg_len), _p(seg_dtype), len(keys), _p(wn), K,
                                     C.c_void_p((table.ctypes.data + 255) // 256 * 256), C.c_size_t(tb), None)
        assert rc == 0
        want = O.fedpavg(models, weights)
        for k, o in zip(keys, outs):
            w = np.asarray(want[k], dtype=np.float32).reshape(-1)
            assert np.array_equal(o[:w.size], w), (k, w.size)
            assert np.all(np.isnan(o[w.size:]))                          # nothing written past the segment
    run()
