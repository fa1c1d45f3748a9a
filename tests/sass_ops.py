"""The SASS of a library cut per kernel (cuobjdump -sass; no GPU needed), shared by the static SASS tests."""
import collections
import re
import subprocess


def kernel_ops(lib):
    """Returns (architectures, {demangled kernel name without its argument list: Counter of opcodes})."""
    sass = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    archs = set(re.findall(r"arch = (sm_\w+)", sass))
    funcs, name = collections.OrderedDict(), None
    for ln in sass.splitlines():
        m = re.search(r"Function : (\S+)", ln)
        if m:
            name = re.sub(r"\(.*", "", subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip())
            funcs[name] = collections.Counter()
        elif name:
            m = re.match(r"\s+/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)", ln)
            if m:
                funcs[name][m.group(1)] += 1
    return archs, funcs
