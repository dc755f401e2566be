"""GPU tuning helper: stage times and the RANSAC iteration histogram of the benchmark sequence."""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from epivo_b200 import api, synth

frames = int(sys.argv[1]) if len(sys.argv) > 1 else 4541
seq = synth.make_sequence(frames, 2000, seed=synth.seed_for(3, 0))
ctx = api.Context(0)
pipe = api.SequencePipeline(seq.n_frames, 2000, ctx=ctx)
pipe.upload(seq.kps, seq.descs)
prm = api.default_params(seq.K.astype(np.float32), threshold=float(os.environ.get("THR", "1.0")),
                         method=api.LMEDS if os.environ.get("LMEDS") else api.RANSAC)
for _ in range(3):
    pipe.run(prm, 0, seq.n_pairs)
acc = np.zeros(16)
for _ in range(5):
    pipe.run(prm, 0, seq.n_pairs)
    acc += pipe.stage_ms()
res = pipe.download(0, seq.n_pairs)
it = res["ransac_iters"]
names = ["total", "match", "presolve", "essential", "pose", "lm", "finish", "match_kernel"]
print({k: round(float(acc[i] / 5), 3) for i, k in enumerate(names)})
import signal; signal.signal(signal.SIGPIPE, signal.SIG_DFL)
print("iters: mean %.2f  <=8 %.3f  <=12 %.3f  <=16 %.3f  <=24 %.3f  <=32 %.3f  max %d" %
      (it.mean(), (it <= 8).mean(), (it <= 12).mean(), (it <= 16).mean(), (it <= 24).mean(), (it <= 32).mean(), it.max()))
print("models/pair mean %.1f" % res["n_models"].mean())
