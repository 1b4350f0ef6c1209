"""Why two builds' transcripts differ: per-frame argmax and best-minus-second margin of the fp32 model's logits
(vasr_forward) on one of bench.py's input sets, and a comparison of two such records.
    VASR_LIB=<a.so> python tools/argmax_margins.py save A.npz [--set S]
    VASR_LIB=<b.so> python tools/argmax_margins.py save B.npz [--set S]
    python tools/argmax_margins.py compare A.npz B.npz [DUMP_A DUMP_B]
bench.py --steps K --dump-outputs D dumps the last timed step, which ran on input set (K - 1) % 4.  compare lists every
frame whose argmax differs between the records with its margin in both, and (given the dumps) every utterance whose
token list differs; a difference is explained when all frames that differ have a margin <= 1e-4."""
import argparse, os, sys
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEAR = 1e-4


def save(out, input_set):
    sys.path.insert(0, os.path.join(ROOT, "velocity-asr_b200"))
    import torch
    import velocity_asr as va
    B, S = 64, 16000 * 15                          # bench.py's workload and seeds
    torch.manual_seed(0)
    model = va.VELOCITYASR(va.VelocityASRConfig(scan_mode="sequential")).cuda().eval()
    g = torch.Generator().manual_seed(1234 + input_set)
    pcm = (torch.randn(B, S, generator=g) * 0.1).cuda()
    with torch.no_grad():
        logits = model(va.compute_mel_spectrogram(pcm))
        top = logits.topk(2, dim=-1).values
        arg = logits.argmax(-1)
    np.savez(out, argmax=arg.cpu().numpy().astype(np.int16), margin=(top[..., 0] - top[..., 1]).cpu().numpy(),
             lib=os.environ.get("VASR_LIB", "libvasr.so"))
    print(f"{out}: {tuple(arg.shape)} frames from {os.environ.get('VASR_LIB', 'libvasr.so')}")


def compare(a_path, b_path, dumps):
    a, b = np.load(a_path), np.load(b_path)
    diff = np.argwhere(a["argmax"] != b["argmax"])
    print(f"frames: {a['argmax'].size}, argmax differs at {len(diff)}")
    worst = 0.0
    for u, t in diff:
        ma, mb = float(a["margin"][u, t]), float(b["margin"][u, t])
        worst = max(worst, min(ma, mb))
        print(f"  utt {u:2d} frame {t:4d}: {int(a['argmax'][u, t]):4d} vs {int(b['argmax'][u, t]):4d}, "
              f"margin {ma:.3g} / {mb:.3g}")
    print(f"largest margin of a differing frame: {worst:.3g} ({'all' if worst <= NEAR else 'NOT all'} <= {NEAR:g})")
    if dumps:
        ta, tb = (np.load(os.path.join(d, "tokens.npy")) for d in dumps)
        rows = np.load(os.path.join(dumps[0], "rows.npy")).astype(int)
        utts = sorted(set(int(u) for u in diff[:, 0]))
        changed = [int(rows[i]) for i in range(len(rows)) if not np.array_equal(ta[i], tb[i])]
        print(f"token lists differ for utterances {changed}; utterances with a differing frame: {utts}; "
              f"{'all' if set(changed) <= set(utts) else 'NOT all'} explained")


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    sp = ap.add_subparsers(dest="cmd", required=True)
    s = sp.add_parser("save"); s.add_argument("out"); s.add_argument("--set", type=int, default=0)
    c = sp.add_parser("compare"); c.add_argument("a"); c.add_argument("b"); c.add_argument("dumps", nargs="*")
    args = ap.parse_args()
    if args.cmd == "save":
        save(args.out, args.set)
    else:
        compare(args.a, args.b, args.dumps)
