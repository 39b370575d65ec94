"""Decode from a token prefix: 50-step decode of B = 64 images at the full geometry (fp16), uniform prefixes n in
{32, 64, 128, 256, 512} and one mixed batch cycling through them.  Images/s from CUDA events around graph replays after warm-up,
per-kernel-class milliseconds from one eager profiled decode, and the card's name and power limit read in the same run.

    python profiles/prefix_bench.py [out.json]          (default prefix_bench.json in the current directory)
"""
import json
import os
import subprocess
import sys

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from selftoktokenizer_b200 import capi, config as C, schedule as S, synth  # noqa: E402

B, REPS, NS = 64, 3, (32, 64, 128, 256, 512)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name(0)


def timed(eng, tok, noise, n):
    eng.set_use_graph(True)
    x = eng.decode(tok, noise, n_tokens=n)                                # capture + warm-up
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(REPS):
        eng.decode(tok, noise, n_tokens=n)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / REPS
    eng.set_use_graph(False)
    eng.set_profile(True)
    eng.decode(tok, noise, n_tokens=n)
    prof = {k: round(v[0], 2) for k, v in eng.get_profile().items()}
    eng.set_profile(False)
    return x, {"ms_per_decode": round(ms, 2), "images_per_s": round(B * 1000.0 / ms, 2), "eager_profile_ms": prof}


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else "prefix_bench.json"
    dev = torch.device("cuda:0")
    d = C.FULL
    eng = capi.Engine(d, synth.synth_state_dict(d, device=dev), device=dev, precision="fp16")
    tok = torch.randint(0, d.codebook_size, (B, d.K), generator=torch.Generator().manual_seed(0)).to(dev)
    noise = synth.synth_tensor("prefix_bench.noise", (B, d.in_channels, d.latent, d.latent), "emb", 1.0, device=dev)
    k = S.make_tables(d.K, d.stages, d.k_per_stage, 50).k
    res = {"card": card(), "batch": B, "precision": "fp16", "steps": 50, "uniform": {}}
    for n in NS:
        x, r = timed(eng, tok, noise, n)
        r["joint_rows_per_decode"] = int(sum(min(int(ki) + 1, n) + 256 for ki in k))
        res["uniform"][str(n)] = r
        if n == d.K:
            eng.set_use_graph(True)
            res["n512_bitwise_equal_to_decode"] = bool(torch.equal(x, eng.decode(tok, noise)))
            assert res["n512_bitwise_equal_to_decode"]
    mixed = [NS[i % len(NS)] for i in range(B)]
    _, res["mixed"] = timed(eng, tok, noise, mixed)
    res["mixed"]["n"] = "cycle " + ",".join(map(str, NS))
    # the mixed batch runs its GEMMs on n_max = 512 context rows; only attention skips the hidden keys
    res["mixed_vs_uniform_512"] = round(res["mixed"]["ms_per_decode"] / res["uniform"]["512"]["ms_per_decode"], 3)
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    json.dump(res, open(out, "w"), indent=1)
    print(json.dumps(res))
    eng.close()


if __name__ == "__main__":
    main()
