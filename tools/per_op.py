import json, sys, collections, os, tempfile
ops = json.load(open(sys.argv[1] if len(sys.argv) > 1 else os.path.join(tempfile.gettempdir(), "ivid_per_op_profile_c2.json")))
agg = collections.OrderedDict()
for label, note, ms, fl, *rest in ops:
    if not label.startswith("conv"): continue
    a = agg.setdefault(note, [0, 0.0, 0.0]); a[0] += 1; a[1] += ms; a[2] += fl
tot = sum(a[1] for a in agg.values())
print(f"{'conv shape':44s} {'n':>3s} {'ms':>8s} {'TF/s':>8s} {'share':>6s}")
for k, a in sorted(agg.items(), key=lambda kv: -kv[1][1]):
    print(f"{k:44s} {a[0]:3d} {a[1]:8.3f} {a[2]/a[1]/1e9:8.1f} {100*a[1]/tot:5.1f}%")
print("total conv ms", round(tot, 3))

gn = collections.OrderedDict()
for label, note, ms, fl, *rest in ops:
    if label != "gn_apply": continue
    a = gn.setdefault(note, [0, 0.0, 0.0]); a[0] += 1; a[1] += ms; a[2] += (rest[0] if rest else 0)
tg = sum(a[1] for a in gn.values())
print(f"\n{'gn_apply shape':44s} {'n':>3s} {'ms':>8s} {'GB/s':>8s} {'share':>6s}")
for k, a in sorted(gn.items(), key=lambda kv: -kv[1][1]):
    print(f"{k:44s} {a[0]:3d} {a[1]:8.3f} {a[2]/a[1]/1e6:8.1f} {100*a[1]/tg:5.1f}%")
print("total gn_apply ms", round(tg, 3), "GB", round(sum(a[2] for a in gn.values())/1e9, 2))

print()
for label, note, ms, fl, *rest in ops:
    if label in ("embed", "pack_input", "attention", "gn_stats"): print(f"{label:12s} {note:40s} {ms:8.3f} ms")
