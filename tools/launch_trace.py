"""Launch trace: every call into libegom2p_b200.so that a fixed set of model cases makes, one JSON line per call, so that
two trees can be compared with `diff`. A change that claims to leave every kernel launch as it was -- a refactor of the
Python glue -- shows an empty diff against its parent.

Recorded per call: the function name; every integer and float argument; for each pointer argument null, or "@j" with j
the position of the first argument of the same call that holds the same address (aliasing such as addend == C_f32,
which selects the GEMM's split-K path, stays visible; raw addresses, which change from run to run, are not recorded);
the non-pointer fields of the PlanDesc / EmbedDesc structs passed by reference; the contents of host integer arrays.

Cases, on the tiny models of tests/test_model_gpu.build_model (swiglu / no-bias family) and
tests/test_gelu_family_gpu.build_gelu (GELU / bias family) with seeded weights, batches and a fixed decoder modality
order, each on a fresh model (so the first casts of the bf16 operands are part of the trace):
  * one training step (forward + backward) for each family, batch (dense; ragged, packed; ragged with pack_rows = False)
    and freeze configuration (nothing, freeze_shared_params(), freeze_encoder(True), encoder + decoder_proj_context,
    decoder[0]; GELU family: also every bias); the causal decoder variant;
  * forward_encoder; forward_decoder with context and with N = 0; one guided GenerationSampler.forward_hidden step
    whose unconditional branch is empty.

    python tools/launch_trace.py --out /tmp/trace_new.jsonl
    python tools/launch_trace.py --root /path/to/parent/tree --out /tmp/trace_old.jsonl
    diff /tmp/trace_old.jsonl /tmp/trace_new.jsonl

--root names the tree whose egom2p_b200 package (with its built library) is traced; the test helpers that build the
cases always come from this tree. Prints the number of calls and of kernel launches per case.
"""
import argparse
import ctypes as C
import json
import os
import random
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

MODS4 = ["tok_cam", "tok_depth", "tok_gaze", "tok_rgb"]
N_ENC, N_DEC = 64, 48
BATCHES = {   # the batches of tests/test_frozen_gpu.py: "dense" fills both budgets, "ragged" gets packed
    "dense": dict(B=2, n_in={"tok_cam": [8, 8], "tok_depth": [24, 24], "tok_gaze": [8, 8], "tok_rgb": [24, 24]},
                  n_tgt={"tok_cam": [6, 6], "tok_depth": [18, 18], "tok_gaze": [6, 6], "tok_rgb": [18, 18]}),
    "ragged": dict(B=4, n_in={"tok_cam": [5, 1, 30, 2], "tok_depth": [30, 10, 0, 1], "tok_gaze": [4, 0, 30, 0], "tok_rgb": [25, 40, 4, 3]},
                   n_tgt={"tok_cam": [10, 30, 0, 1], "tok_depth": [20, 0, 40, 0], "tok_gaze": [3, 0, 0, 0], "tok_rgb": [15, 18, 70, 4]}),
}


def _freeze(*params):
    for p in params:
        p.requires_grad = False


FREEZE = {
    "none": lambda m: None,
    "shared": lambda m: m.freeze_shared_params(),
    "encoder": lambda m: m.freeze_encoder(freeze_embeddings=True),
    "encoder_and_context": lambda m: (m.freeze_encoder(freeze_embeddings=True), _freeze(*m.decoder_proj_context.parameters())),
    "decoder0": lambda m: _freeze(*m.decoder[0].parameters()),
    "biases": lambda m: _freeze(*[p for n, p in m.named_parameters() if n.endswith(".bias")]),
}


class Recorder:
    """Stands in for the loaded library (egom2p_b200._lib._lib): records every egom2p_* call, then makes it."""

    def __init__(self, lib):
        self.lib, self.calls = lib, []

    def __getattr__(self, name):
        fn = getattr(self.lib, name)
        if not name.startswith("egom2p_"):
            return fn

        def call(*args):
            self.calls.append((name, record(fn.argtypes, args)))
            return fn(*args)
        return call


def _address(a):
    return a.value if isinstance(a, C.c_void_p) else (a or None)


def record(argtypes, args):
    addr = [_address(a) if t is C.c_void_p else None for t, a in zip(argtypes, args)]
    out = []
    for t, a, p in zip(argtypes, args, addr):
        if t is C.c_void_p:
            out.append(None if p is None else f"@{addr.index(p)}")
        elif isinstance(a, C.Array):            # host integer array (plan_rows' modality ids)
            out.append(list(a))
        elif hasattr(a, "_obj"):                # C.byref(PlanDesc / EmbedDesc): the non-pointer fields
            fields = {}
            for f, ft in a._obj._fields_:
                if getattr(ft, "_type_", ft) is not C.c_void_p:
                    v = getattr(a._obj, f)
                    fields[f] = list(v) if isinstance(v, C.Array) else v
            out.append(fields)
        else:
            out.append(a)
    return out


def build_cases(torch):
    import gelu_oracle as go
    import synth
    from test_gelu_family_gpu import build_gelu
    from test_model_gpu import build_model, to_cuda
    random.seed(3)
    order = random.sample(MODS4, len(MODS4))
    families = {
        "swiglu": (synth.make_cfg(192, 3, 2, 2, MODS4, video_vocab=512, video_thw=(5, 4, 4)), synth.make_state_dict, build_model),
        "gelu": (go.make_cfg(384, 6, 2, 2, MODS4, video_vocab=512, video_thw=(5, 4, 4)), go.make_state_dict, build_gelu),
    }

    def model(fam, causal=False):
        cfg, make_sd, build = families[fam]
        cfg = dict(cfg, causal=causal)
        m = build(cfg).cuda()
        m.load_state_dict(make_sd(cfg, 5), strict=True)
        m.fixed_decoder_order = list(order)
        return m, cfg

    def train(fam, batch, pack_rows, freeze, causal=False):
        def run():
            m, cfg = model(fam, causal)
            m.pack_rows = pack_rows
            FREEZE[freeze](m)
            loss, _ = m(to_cuda(synth.make_batch(cfg, seed=11, **BATCHES[batch])), N_ENC, N_DEC)
            loss.backward()
        return run

    def rand(*shape):
        return torch.randn(*shape, generator=torch.Generator().manual_seed(7)).cuda()

    def encoder(fam):
        def run():
            m, cfg = model(fam)
            mask = torch.arange(N_ENC)[None, None, :] >= torch.tensor([N_ENC, 37])[:, None, None]
            m.forward_encoder(rand(2, N_ENC, cfg["dim"]), encoder_mask=mask.cuda())
        return run

    def decoder(fam, n_ctx):
        def run():
            m, cfg = model(fam)
            mask = torch.arange(n_ctx)[None, None, :] >= torch.tensor([n_ctx, n_ctx // 2])[:, None, None]
            m.forward_decoder(rand(2, N_DEC, cfg["dim"]), rand(2, n_ctx, cfg["dim"]), encoder_mask=mask.cuda() if n_ctx else None,
                              decoder_attention_mask=None)
        return run

    def guided_step(fam):   # tests/test_gelu_family_gpu.test_forward_hidden_guided_step_against_oracle
        def run():
            from egom2p_b200.generate import GenerationSampler
            m, _ = model(fam)
            B, L = 1, 80
            ids = torch.randint(0, 512, (B, 5, 4, 4), generator=torch.Generator().manual_seed(0))
            md = {"tok_rgb": {"tensor": ids.cuda(), "input_mask": torch.zeros(B, L, dtype=torch.bool).cuda(),
                              "target_mask": torch.ones(B, L, dtype=torch.bool).cuda()},
                  "tok_cam": {"tensor": torch.zeros(B, 30, dtype=torch.int64).cuda(), "input_mask": torch.ones(B, 30, dtype=torch.bool).cuda(),
                              "target_mask": torch.zeros(B, 30, dtype=torch.bool).cuda()}}
            GenerationSampler(m.eval()).forward_hidden(md, "tok_cam", ["tok_rgb"], {"tok_rgb": [L], "tok_cam": [0]},
                                                       torch.tensor([[7, 11, 29, 5, 20]]).cuda())
        return run

    cases = {}
    for fam in families:
        for batch, pack_rows in (("dense", True), ("ragged", True), ("ragged", False)):
            for freeze in FREEZE:
                if freeze != "biases" or fam == "gelu":
                    cases[f"train/{fam}/{batch}{'' if pack_rows else '_unpacked'}/{freeze}"] = train(fam, batch, pack_rows, freeze)
    cases["train/swiglu/ragged/none/causal"] = train("swiglu", "ragged", True, "none", causal=True)
    for fam in families:
        cases[f"forward_encoder/{fam}"] = encoder(fam)
        cases[f"forward_decoder/{fam}"] = decoder(fam, N_ENC)
        cases[f"forward_decoder_no_context/{fam}"] = decoder(fam, 0)
        cases[f"forward_hidden_guided/{fam}"] = guided_step(fam)
    return cases


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=ROOT, help="tree whose egom2p_b200 package is traced (default: this one)")
    ap.add_argument("--out", required=True, help="JSON lines, one per library call")
    args = ap.parse_args()
    for p in (os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests"), os.path.abspath(args.root)):
        sys.path.insert(0, p)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("launch_trace.py runs the cases on the GPU; no CUDA device found")
    from egom2p_b200 import _lib
    rec = Recorder(_lib.load())
    _lib._lib = rec
    summary = []
    with open(args.out, "w") as f:
        for name, run in build_cases(torch).items():
            rec.calls.clear()
            l0 = rec.lib.egom2p_launch_count()
            with torch.no_grad() if not name.startswith("train/") else torch.enable_grad():
                run()
            torch.cuda.synchronize()
            launches = rec.lib.egom2p_launch_count() - l0
            for i, (fn, a) in enumerate(rec.calls):
                f.write(json.dumps({"case": name, "i": i, "fn": fn, "args": a}, separators=(",", ":")) + "\n")
            summary.append({"case": name, "calls": len(rec.calls), "launches": launches})
    print(json.dumps({"package": os.path.dirname(_lib.__file__), "cases": summary}, indent=1))


if __name__ == "__main__":
    main()
