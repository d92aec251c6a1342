"""`deepconsensus_b200.run` on the reference's BAM fixtures (7 of its 10 ZMWs, 958 windows), seeded weights: stage times.
--use_ccs_smart_windows: the same subreads with ccs_wl.bam (seeded `wl` tags), windows from the tags."""
import json, os, shutil, sys, tempfile, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deepconsensus_b200 import run as run_lib
g = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
tmp = tempfile.mkdtemp()
shutil.copytree(os.path.join(g, "ckpt", "model"), os.path.join(tmp, "model"))
smart = "--use_ccs_smart_windows" in sys.argv[1:]
kw = dict(use_ccs_smart_windows=True) if smart else {}
for out in ("out.fastq", "out.bam"):
  t0 = time.time()
  c = run_lib.run(subreads_to_ccs=os.path.join(g, "human_1m", "subreads_to_ccs.bam"), ccs_bam=os.path.join(g, "human_1m", "ccs_wl.bam" if smart else "ccs.bam"),
                  checkpoint=os.path.join(tmp, "model", "checkpoint-1"), output=os.path.join(tmp, out), batch_zmws=100,
                  batch_size=1024, min_quality=0, random_weights=3, **kw)
  st = json.load(open(os.path.join(tmp, out + ".inference.json")))
  print(out, "wall %.2f s (incl. engine creation)" % (time.time() - t0), json.dumps(st))
