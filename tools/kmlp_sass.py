"""Prints the SASS of every k_mlp_tc instance in `cuobjdump -sass` listings, sorted by name, for comparing two builds.
With --only FILE, only the instances named in FILE (e.g. the previous build's list)."""
import re, sys
args = sys.argv[1:]
only = None
if args[0] == "--only":
    only = set(open(args[1]).read().split()); args = args[2:]
funcs = {}
for path in args:
    cur = None
    for line in open(path):
        m = re.match(r'\s*Function : (\S+)', line)
        if m:
            cur = m.group(1) if 'k_mlp_tc' in m.group(1) else None
            if cur: funcs[cur] = []
        elif cur:
            funcs[cur].append(line)
for k in sorted(funcs):
    if only is None or k in only:
        sys.stdout.write("Function : %s\n" % k); sys.stdout.writelines(funcs[k])
