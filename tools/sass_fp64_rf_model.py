"""Static model of K1's RK4 stage loop from its SASS (cuobjdump -sass of fk.o, the fk_rk4_fp64_kernel<6,1> function):

  * the scheduled stall counts (control codes) of the loop body: the time ONE warp needs per stage if nothing else
    ran -- against the 2 cycles per FP64 warp instruction the pipe needs;
  * the register-file read model of the FP64 pipe: an instruction's issue cost is max(2, distinct 64-bit register
    sources that are not served by the operand reuse cache) -- a DFMA with three distinct register pairs needs three
    reads from each of the two register banks, i.e. 3 cycles, not 2 (B300_MICROARCH.md, "RF banking": rt =
    max(rt_pipe, #even_distinct, #odd_distinct)).  The ratio of the two sums is the ceiling of
    sm__pipe_fp64_cycles_active for this instruction stream.

usage:  cuobjdump -sass interactive-rate-tendons_b200/csrc/fk.o | awk '/Function :.*fk_rk4_fp64_kernelILi6ELb1E/{f=1}
        f&&/Function :/&&!/fk_rk4_fp64_kernelILi6ELb1E/{f=0} f' > /tmp/fk.sass;  python tools/sass_fp64_rf_model.py /tmp/fk.sass
"""
import re
import sys
from collections import Counter

FP64 = re.compile(r'(DFMA|DMUL|DADD|DSETP)')


def parse(path):
    lines = open(path).read().split('\n')
    ins, i = [], 0
    while i < len(lines):
        m = re.match(r'\s*/\*([0-9a-f]+)\*/\s+(.*?);\s*/\* (0x[0-9a-f]+) \*/', lines[i])
        if m and i + 1 < len(lines):
            m2 = re.match(r'\s*/\* (0x[0-9a-f]+) \*/', lines[i + 1])
            if m2:
                hi = int(m2.group(1), 16)
                ins.append((int(m.group(1), 16), m.group(2).strip(), (hi >> 41) & 0xf))   # address, text, stall count
                i += 2
                continue
        i += 1
    return ins


def stage_loops(ins):
    """the innermost loops that hold one derivative evaluation: a backward branch whose body has NT + 1 = 7 rsqrt
    seeds (6 tendons and |v|) -- the generic stage loop (routing through a pointer) and, when built, the fast-path
    loop (routing from constant memory through uniform registers)"""
    addr = {a: k for k, (a, _, _) in enumerate(ins)}
    out = []
    for k, (a, txt, _) in enumerate(ins):
        m = re.search(r'BRA.*0x([0-9a-f]+)', txt)
        if not m:
            continue
        t = int(m.group(1), 16)
        if t < a and t in addr:
            body = ins[addr[t]:k + 1]
            if sum(1 for x in body if 'MUFU.RSQ64H' in x[1]) == 7:
                out.append(body)
    if not out:
        raise SystemExit("stage loop not found")
    return out


def report(body):
    ops = Counter()
    two = rf = stall = 0
    reads = Counter()
    kept = {}                      # operand slot -> register held by the reuse cache
    for _, txt, st in body:
        stall += st
        t = re.sub(r'^@!?U?P\d\s+', '', txt)
        op = t.split()[0]
        ops[op.split('.')[0]] += 1
        if not FP64.match(op):
            kept = {}              # conservative: any other instruction in between drops the cached operands
            continue
        regs, keep = [], {}
        for slot, o in enumerate(t[len(op):].split(',')[1:]):
            m = re.search(r'\bR(\d+)(\.reuse)?', o)     # UR.. / c[..] / immediates do not read the register file
            if not m:
                continue
            r = int(m.group(1))
            if m.group(2):
                keep[slot] = r
            if kept.get(slot) != r:
                regs.append(r)
        n = len(set(regs))
        reads[(op.split('.')[0], n)] += 1
        two += 2
        rf += max(2, n)
        kept = keep
    nf = sum(reads.values())
    print("loop at 0x%x: %d instructions, %d FP64 (%s)" % (body[0][0], len(body), nf,
                                                          ", ".join("%s %d" % kv for kv in ops.most_common(7))))
    print("  one warp alone (sum of scheduled stall counts): %d cycles per stage" % stall)
    print("  FP64 pipe cycles per stage and warp: %d at 2 per instruction, %d with the register-read model -> ceiling "
          "of pipe_fp64_cycles_active %.1f %%" % (two, rf, 100.0 * two / rf))
    print("  distinct register-pair reads per instruction:", sorted(reads.items()))


def main():
    for body in stage_loops(parse(sys.argv[1])):
        report(body)


if __name__ == "__main__":
    main()
