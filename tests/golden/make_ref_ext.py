"""Record what the reference's own CUDA extensions return on the inputs of tests/test_gpu_reference_ext.py.

Needs a GPU and the two extensions ``oracle/build_ref.py`` builds from the original project into ``oracle/_ref/``:
    python oracle/build_ref.py
    python tests/golden/make_ref_ext.py [OUT.npz]      # default: tests/golden/ref_ext.npz

Per case the file holds a SHA-256 of the inputs, a SHA-256 and a fixed sample of every output the test compares
bit for bit, the gradient reductions whole, and a fixed sample of every GPTQ output.
"""
import importlib.util
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import test_gpu_reference_ext as T  # noqa: E402


def load(name):
    path = os.path.join(ROOT, "oracle", "_ref", name + ".so")
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def bits_record(out, key, a):
    a = np.asarray(a, np.float32).reshape(-1)
    out[key + "_sha256"] = np.array(T.digest(a))
    out[key + "_sample"] = a[T.sample_index(a.size, T.BITS_SAMPLE)]


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "ref_ext.npz")
    fq, gq = load("fake_quant_ref"), load("gptq_ref")
    out = {}
    for case in T.PERTENSOR_CASES:
        key = T.pertensor_key(*case)
        qmin, qmax = case[1:3]
        x, gy, s, z = T.pertensor_inputs(*case)
        out[key + "_inputs_sha256"] = np.array(T.digest(x, gy, s, z))
        xt, gt, st, zt = T.t(x), T.t(gy), T.t(s).requires_grad_(True), T.t(z).requires_grad_(True)
        bits_record(out, key + "_y", fq.quant_pertensor_forward(xt, st, zt, qmin, qmax, 0).cpu().numpy())
        gx, gs, gz = T._np(*fq.quant_pertensor_backward(xt, st, zt, gt, qmin, qmax, 0))
        bits_record(out, key + "_gx", gx)
        out[key + "_gs"], out[key + "_gz"] = gs, gz
    for case in T.PERCHANNEL_CASES:
        key = T.perchannel_key(*case)
        ch_axis, qmin, qmax = case[1:]
        x, gy, s, z = T.perchannel_inputs(*case)
        out[key + "_inputs_sha256"] = np.array(T.digest(x, gy, s, z))
        xt, gt, st, zt = T.t(x), T.t(gy), T.t(s).requires_grad_(True), T.t(z).requires_grad_(True)
        bits_record(out, key + "_y", fq.quant_perchannel_forward(xt, st, zt, qmin, qmax, ch_axis, 0).cpu().numpy())
        gx, gs, gz = T._np(*fq.quant_perchannel_backward(xt, st, zt, gt, qmin, qmax, ch_axis, 0))
        bits_record(out, key + "_gx", gx)
        out[key + "_gs"], out[key + "_gz"] = gs, gz
    x, gy, s, z = T.gate_inputs()
    out["gate_inputs_sha256"] = np.array(T.digest(x, gy, s, z))
    gates = []
    for rs, rz in T.GATE_CASES:
        _, gs, gz = fq.quant_pertensor_backward(T.t(x), T.t(s).requires_grad_(rs), T.t(z).requires_grad_(rz), T.t(gy), -8, 7, 0)
        gates.append((float(gs), float(gz)))
    out["gate_gs"], out["gate_gz"] = np.float32(gates).T
    for case in T.GPTQ_CASES:
        key = T.gptq_key(*case)
        bit, m, k, n, gs = case
        x, qw, scales, zeros, bias = T.gptq_inputs(*case)
        out[key + "_inputs_sha256"] = np.array(T.digest(*T._np(x, qw, scales, zeros, bias)))
        y = bias.expand(m, n).contiguous()
        if gs == -1:
            getattr(gq, T.gptq_name(bit, gs))(x, qw, y, scales, zeros)
        else:
            getattr(gq, T.gptq_name(bit, gs))(x, qw, y, scales, zeros, gs)
        out[key + "_y_sample"] = y.cpu().numpy().reshape(-1)[T.sample_index(m * n, T.GPTQ_SAMPLE)]
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes,", torch.cuda.get_device_name())


if __name__ == "__main__":
    main()
