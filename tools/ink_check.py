import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from flow_check import make, gen, time_steps
ref, embed = make({"CTB_NO_FLOW": "1"})
a, _ = make({"CTB_FLOW_NO_INK": "1"})
b, _ = make({})
ok = True
for B, greedy, steps in ((1, True, 80), (2, False, 70), (1, False, 130), (2, True, 40)):
    lengths = [16, 7][:B]
    r = gen(ref, embed, lengths, steps, greedy)
    x = gen(a, embed, lengths, steps, greedy)
    y = gen(b, embed, lengths, steps, greedy)
    for i in range(B):
        e1, e2 = torch.equal(r.ids[i], x.ids[i]), torch.equal(r.ids[i], y.ids[i])
        hd = float((r.hiddens[i] - y.hiddens[i]).abs().max())
        print(f"B={B} greedy={greedy} row {i}: noink_equal={e1} ink_equal={e2} n={len(y.ids[i])} |dh|={hd:.2e}", flush=True)
        if not e2:
            d = (r.ids[i] != y.ids[i]).any(-1).float().argmax()
            print("   first diff step", int(d), r.ids[i][int(d)].tolist(), y.ids[i][int(d)].tolist())
        ok &= e1 and e2
# early finish (EOS allowed): min_new small
from chattts_b200.processors import gen_logits
from chattts_b200.prompts import synth_prompt_batch
ids, mask, tmask = synth_prompt_batch([16, 9], seed=3)
warp, proc = gen_logits(num_code=625, top_P=0.7, top_K=20, repetition_penalty=1.05)
outs = []
for gmod in (ref, b):
    o = list(gmod.generate(embed(ids, tmask), ids, temperature=torch.tensor([1.5] * 4), eos_token=625, attention_mask=mask,
                           max_new_token=200, min_new_token=2, logits_processors=(*proc, *warp), return_hidden=False,
                           show_tqdm=False, manual_seed=7))[-1]
    outs.append(o)
print("EOS run lens:", [len(t) for t in outs[0].ids], [len(t) for t in outs[1].ids],
      "equal:", [bool(torch.equal(outs[0].ids[i], outs[1].ids[i])) for i in range(2)], flush=True)
print("INK PARITY", "OK" if ok else "MISMATCH", flush=True)
print("old k_step B=1 %.1f us/step" % time_steps(ref, embed, 1, 512))
print("flow no-ink B=1 %.1f  B=2 %.1f" % (time_steps(a, embed, 1, 512), time_steps(a, embed, 2, 512)))
print("flow ink    B=1 %.1f  B=2 %.1f" % (time_steps(b, embed, 1, 512), time_steps(b, embed, 2, 512)), flush=True)

import ctypes as C
from chattts_b200 import _lib
tr, _ = make({"CTB_MEGA_TRACE": "1"})
time_steps(tr, embed, 1, 64, reps=1)
buf = (C.c_ulonglong * 4096)()
_lib.check(_lib.load().ctb_gpt_debug_trace(tr._handle, buf, 4096))
t = [int(buf[i]) for i in range(110)]
# stamps: 0 launch start, 1 table+issue, 2 input staged, 3..102 the 100 phases, 103 heads, 104 sampler CTA done, 105 ids polled + bookkeeping
sk = [int(buf[3100 + i]) for i in range(8)]
print("sampler cycles: temp/pen+max=%d den=%d sort=%d scan+nrem=%d ban+den2=%d argmax=%d total=%d" % (
    sk[1] - sk[0], sk[2] - sk[1], sk[3] - sk[2], sk[4] - sk[3], sk[5] - sk[4], sk[6] - sk[5], sk[6] - sk[0]), flush=True)
print("step breakdown ns: table+issue=%d input=%d layers=%d (layer0 phaseA=%d) heads=%d sampler=%d idx+finalize=%d total=%d" % (
    t[1] - t[0], t[2] - t[1], t[102] - t[2], t[3] - t[2], t[103] - t[102], t[104] - t[103], t[105] - t[104], t[105] - t[0]), flush=True)
