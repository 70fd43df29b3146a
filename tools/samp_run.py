import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from volcano_b200 import engine
from volcano_b200.synth import make_snapshot
snap = make_snapshot("cfg2")
snap.conf.percentage_nodes_to_find = 0
e = engine.Engine(snap); e.upload()
for _ in range(2):
    r = e.allocate()
print("sampling cfg2:", len(r.decisions), r.stats["commit_ms"], "ms", len(r.decisions)/r.stats["commit_ms"]*1e3, "pods/s", "last", r.stats["last_processed_node_index"])
e.close()
