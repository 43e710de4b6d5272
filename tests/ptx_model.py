"""A CPU model of the inline PTX of the device field core (schnorr-sig_b200/csrc/fp.cuh).

The host build of fp.cuh replaces every asm block with a portable fallback, so the CPU suite never runs the
instruction sequences the kernels run.  This module preprocesses fp.cuh as the device compiler sees it
(`__CUDA_ARCH__` defined), extracts every `asm(...)` block with the function around it,
and interprets the instructions on 32-bit words with one carry flag (CC.CF; a borrow for sub/subc).  Operands are
bound by the C expressions of the constraint lists, not by position, so a block that passes a subset of its
function's words is modelled correctly.  `FpCore` mirrors the C around the asm blocks, so it predicts the exact words
the device returns.  An instruction outside the modelled subset is an error: a new instruction in fp.cuh makes
the model fail until it is extended.
"""
import functools
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FP_CUH = os.path.join(ROOT, "schnorr-sig_b200", "csrc", "fp.cuh")

M32 = 0xFFFFFFFF
M64 = (1 << 64) - 1
P = 0xFFFFFFFF00000001

# every function of fp.cuh that holds an asm block under __CUDA_ARCH__
MODELLED = ("fp_sub", "fp_reduce96_nc", "fp_reduce160_t", "wide_mac", "wide_mac_sqr", "wide_reduce_t", "wide_add64",
            "fp_mul_nc", "fp_sqr_nc", "fp_mul7_nc")


class ModelError(Exception):
    pass


@functools.lru_cache(maxsize=None)
def device_source():
    """fp.cuh as the device compiler sees it (namespace sb only)."""
    out = subprocess.check_output(["g++", "-E", "-P", "-x", "c++", "-D__CUDACC__", "-D__CUDA_ARCH__=1000", FP_CUH],
                                  text=True, stderr=subprocess.DEVNULL)   # "#pragma once in main file"
    return out[out.index("namespace sb"):]


def _split_top(text, sep):
    """Split at `sep` outside string literals and parentheses."""
    parts, depth, cur, i = [], 0, [], 0
    while i < len(text):
        ch = text[i]
        if ch == '"':
            j = i + 1
            while text[j] != '"':
                j += 2 if text[j] == "\\" else 1
            cur.append(text[i:j + 1])
            i = j + 1
            continue
        if ch == "(":
            depth += 1
        elif ch == ")":
            depth -= 1
        if ch == sep and depth == 0:
            parts.append("".join(cur))
            cur = []
        else:
            cur.append(ch)
        i += 1
    parts.append("".join(cur))
    return parts


def _asm_extent(src, start):
    """Index just past the ')' closing the asm( that opens at src[start]."""
    depth, i = 0, start
    while True:
        ch = src[i]
        if ch == '"':
            i += 1
            while src[i] != '"':
                i += 2 if src[i] == "\\" else 1
        elif ch == "(":
            depth += 1
        elif ch == ")":
            depth -= 1
            if depth == 0:
                return i + 1
        i += 1


def _operands(text):
    ops = []
    for part in _split_top(text, ","):
        part = part.strip()
        if not part:
            continue
        m = re.match(r'"([^"]*)"\s*\((.*)\)$', part, re.S)
        if not m:
            raise ModelError("cannot parse asm operand %r" % part)
        ops.append((m.group(1), re.sub(r"\s+", "", m.group(2))))
    return ops


_OPCODES = [
    (re.compile(r"(add|sub)(c?)(\.cc)?\.u32$"), "addsub"),
    (re.compile(r"mul\.(lo|hi)\.u32$"), "mul"),
    (re.compile(r"mad(c?)\.(lo|hi)(\.cc)?\.u32$"), "mad"),
    (re.compile(r"shr\.(s32|u32)$"), "shr"),
    (re.compile(r"shl\.b32$"), "shl"),
    (re.compile(r"shf\.l\.clamp\.b32$"), "shf"),
]


class AsmBlock:
    def __init__(self, function, template, outputs, inputs):
        self.function = function
        self.outputs = outputs          # [(constraint, C expression)]
        self.inputs = inputs
        self.template = template
        self.temps = set()
        self.code = []
        for raw in re.split(r"[;\n]", template):
            line = raw.strip()
            if line in ("", "{", "}"):
                continue
            if line.startswith(".reg"):
                m = re.match(r"\.reg\s+\.(u32|b32)\s+(.*)$", line)
                if not m:
                    raise ModelError("%s: unsupported register declaration %r" % (function, line))
                self.temps.update(n.strip() for n in m.group(2).split(","))
                continue
            opcode, _, rest = line.partition(" ")
            args = [a.strip() for a in rest.split(",")]
            for pattern, kind in _OPCODES:
                m = pattern.match(opcode)
                if m:
                    self.code.append((kind, m.groups(), args, line))
                    break
            else:
                raise ModelError("%s: instruction %r is not modelled" % (function, line))

    def run(self, env):
        """Executes the block; env maps C expressions (whitespace removed) to u32 values.  Returns the values of the
        output expressions."""
        operands = self.outputs + self.inputs
        regs = {}
        for k, (cons, expr) in enumerate(operands):
            if cons.startswith("="):
                regs["%" + str(k)] = None        # written before it is read, or the model fails
            else:
                if expr not in env:
                    raise ModelError("%s: no value bound to operand %s" % (self.function, expr))
                regs["%" + str(k)] = env[expr] & M32
        for t in self.temps:
            regs[t] = None
        cf = [None]

        def val(x):
            if x in regs:
                if regs[x] is None:
                    raise ModelError("%s: %s read before it is written" % (self.function, x))
                return regs[x]
            if re.match(r"^(0x[0-9a-fA-F]+|\d+)$", x):
                return int(x, 0) & M32
            raise ModelError("%s: unknown operand %r" % (self.function, x))

        def carry():
            if cf[0] is None:
                raise ModelError("%s: carry flag read before it is set" % self.function)
            return cf[0]

        for kind, g, args, line in self.code:
            d, src = args[0], [val(a) for a in args[1:]]
            if d not in regs:
                raise ModelError("%s: unknown destination in %r" % (self.function, line))
            if kind == "addsub":
                op, withc, cc = g
                c = carry() if withc else 0
                if op == "add":
                    s = src[0] + src[1] + c
                    out = s >> 32
                else:
                    s = src[0] - src[1] - c
                    out = 1 if s < 0 else 0     # CC.CF holds the borrow after sub/subc
                r = s & M32
            elif kind == "mul":
                p = src[0] * src[1]
                r, cc = (p & M32) if g[0] == "lo" else (p >> 32), None
            elif kind == "mad":
                withc, half, cc = g
                p = src[0] * src[1]
                s = ((p & M32) if half == "lo" else (p >> 32)) + src[2] + (carry() if withc else 0)
                r, out = s & M32, s >> 32
            elif kind == "shr":
                n = min(src[1], 32)
                x = src[0] - (1 << 32) if (g[0] == "s32" and src[0] >> 31) else src[0]
                r, cc = (x >> n) & M32, None
            elif kind == "shl":
                r, cc = (src[0] << min(src[1], 32)) & M32, None
            else:  # shf.l.clamp.b32 d, a, b, n: the high word of (b:a) << min(n, 32)
                r, cc = ((((src[1] << 32) | src[0]) << min(src[2], 32)) >> 32) & M32, None
            regs[d] = r
            if cc:
                cf[0] = out
        res = {}
        for k, (cons, expr) in enumerate(self.outputs):
            res[expr] = val("%" + str(k))
        return res


@functools.lru_cache(maxsize=None)
def asm_blocks():
    """{function name: [AsmBlock]} of the device form of fp.cuh."""
    src = device_source()
    heads = [(m.start(), m.group(1)) for m in re.finditer(r"\b(?:fp_t|void)\s+(\w+)\s*\(", src)]
    blocks = {}
    for m in re.finditer(r"\basm\s*\(", src):
        end = _asm_extent(src, m.end() - 1)
        parts = _split_top(src[m.end():end - 1], ":")
        template = "".join(bytes(s, "ascii").decode("unicode_escape") for s in re.findall(r'"((?:[^"\\]|\\.)*)"', parts[0]))
        outputs = _operands(parts[1]) if len(parts) > 1 else []
        inputs = _operands(parts[2]) if len(parts) > 2 else []
        fn = [name for pos, name in heads if pos < m.start()][-1]
        blocks.setdefault(fn, []).append(AsmBlock(fn, template, outputs, inputs))
    return blocks


def count_asm():
    return len(re.findall(r"\basm\s*\(", device_source()))


def lo(x):
    return x & M32


def hi(x):
    return (x >> 32) & M32


def join(w0, w1):
    return (w1 << 32) | w0


# ---- the paths a reduction takes (the order of fp_reduce160_t) ----------------------------------------------------
def reduce_path(x0, x1, x2, x3=0, x4=0):
    """(m, c, k, t) of the reduction of x0 + x1 2^32 + x2 2^64 + x3 2^96 + x4 2^128: m = 1 when (x1:x0) - (x4:x3)
    borrows, c = 1 when the fold + x2 (2^32 - 1) carries, k = c - m the multiple of EPS applied, t the 64-bit value
    the correction is applied to."""
    a, b = join(x0, x1), join(x3, x4)
    m = 1 if a < b else 0
    f = ((a - b) & M64) + x2 * M32
    c = f >> 64
    return m, c, c - m, f & M64


def product_words(a, b):
    p = a * b
    return tuple((p >> (32 * i)) & M32 for i in range(4))


def product_path(a, b):
    return reduce_path(*product_words(a, b))


def wide_words(state):
    """The words x0..x4 wide_reduce_t hands to fp_reduce160_t."""
    e0, e1, e2, e3, e4, o1, o2, o3 = state
    h = join(e1, e2) | (e3 << 64) | (e4 << 96)
    h += o1 | (o2 << 32) | (o3 << 64)
    return (e0,) + tuple((h >> (32 * i)) & M32 for i in range(4))


def wide_value(state):
    e0, e1, e2, e3, e4, o1, o2, o3 = state
    E = sum(w << (32 * i) for i, w in enumerate((e0, e1, e2, e3, e4)))
    O = sum(w << (32 * i) for i, w in enumerate((o1, o2, o3)))
    return E, O


def wide_state(E, O):
    return tuple((E >> (32 * i)) & M32 for i in range(5)) + tuple((O >> (32 * i)) & M32 for i in range(3))


class FpCore:
    """The device field core, instruction for instruction."""

    def __init__(self):
        self.blocks = asm_blocks()

    def _asm(self, fn, env):
        (block,) = self.blocks[fn]
        return block.run(env)

    def fp_sub(self, a, b):
        r = self._asm("fp_sub", {"a0": lo(a), "a1": hi(a), "b0": lo(b), "b1": hi(b)})
        return join(r["d0"], r["d1"])

    def fp_add(self, a, b):
        return self.fp_sub(a, (P - b) & M64)

    def fp_neg(self, a):
        return (P - a) & M64 if a else 0

    def fp_dbl(self, a):
        return self.fp_add(a, a)

    def fp_reduce96_nc(self, x0, x1, x2):
        r = self._asm("fp_reduce96_nc", {"x0": x0, "x1": x1, "x2": x2})
        return join(r["t0"], r["t1"])

    def fp_canon_sel(self, r):
        t0, t1 = lo(r), hi(r)
        ge = t1 == M32 and t0 != 0
        return join((t0 - 1) & M32 if ge else t0, 0 if ge else t1)

    def fp_reduce96(self, x0, x1, x2):
        return self.fp_canon_sel(self.fp_reduce96_nc(x0, x1, x2))

    def fp_reduce160_t(self, canon, x0, x1, x2, x3, x4):
        env = {"x0": x0, "x1": x1, "x2": x2, "x3": x3, "x4": x4}
        r = self._asm("fp_reduce160_t", env)
        v = join(r["t0"], r["t1"])
        return self.fp_canon_sel(v) if canon else v

    def fp_canon(self, x):
        return x - P if x >= P else x

    def fp_mul_nc(self, a, b):
        r = self._asm("fp_mul_nc", {"a0": lo(a), "a1": hi(a), "b0": lo(b), "b1": hi(b)})
        return join(r["t0"], r["t1"])

    def fp_sqr_nc(self, a):
        r = self._asm("fp_sqr_nc", {"a0": lo(a), "a1": hi(a)})
        return join(r["t0"], r["t1"])

    def fp_mul(self, a, b):
        return self.fp_canon(self.fp_mul_nc(a, b))

    def fp_sqr(self, a):
        return self.fp_canon(self.fp_sqr_nc(a))

    def fp_mul_small(self, a, k):
        lo_, hi_ = lo(a) * k, (a >> 32) * k
        s = (lo_ + (hi_ << 32)) & M64
        c = 1 if s < lo_ else 0
        return self.fp_reduce96(lo(s), hi(s), ((hi_ >> 32) + c) & M32)

    def fp_mul7_nc(self, a):
        r = self._asm("fp_mul7_nc", {"a0": lo(a), "a1": hi(a)})
        return join(r["t0"], r["t1"])

    def fp_sqr_n(self, a, n):
        for _ in range(n):
            a = self.fp_sqr_nc(a)
        return self.fp_canon(a)

    def fp_inv(self, a):
        mul, sqr, sqr_n = self.fp_mul, self.fp_sqr, self.fp_sqr_n
        t2 = mul(sqr(a), a)
        t4 = mul(sqr_n(t2, 2), t2)
        t8 = mul(sqr_n(t4, 4), t4)
        t16 = mul(sqr_n(t8, 8), t8)
        t32 = mul(sqr_n(t16, 16), t16)
        t31 = mul(sqr_n(mul(sqr_n(mul(sqr_n(t16, 8), t8), 4), t4), 2), t2)
        t31 = mul(sqr(t31), a)
        return mul(sqr_n(t31, 33), t32)

    # ---- the accumulator: states are tuples (e0, e1, e2, e3, e4, o1, o2, o3) ----
    @staticmethod
    def _wenv(w):
        return dict(zip(("w.e0", "w.e1", "w.e2", "w.e3", "w.e4", "w.o1", "w.o2", "w.o3"), w))

    @staticmethod
    def _wout(r):
        return tuple(r[k] for k in ("w.e0", "w.e1", "w.e2", "w.e3", "w.e4", "w.o1", "w.o2", "w.o3"))

    def wide_mac(self, w, a, b):
        env = self._wenv(w)
        env.update(a0=lo(a), a1=hi(a), b0=lo(b), b1=hi(b))
        return self._wout(self._asm("wide_mac", env))

    def wide_mac_sqr(self, w, a):
        env = self._wenv(w)
        env.update(a0=lo(a), a1=hi(a))
        return self._wout(self._asm("wide_mac_sqr", env))

    def wide_add64(self, w, v):
        env = self._wenv(w)
        env.update({"(uint32_t)v": lo(v), "(uint32_t)(v>>32)": hi(v)})
        r = self._asm("wide_add64", env)
        return tuple(r[k] for k in ("w.e0", "w.e1", "w.e2", "w.e3", "w.e4")) + tuple(w[5:])

    def wide_double(self, w):
        e0, e1, e2, e3, e4, o1, o2, o3 = w
        return ((e0 << 1) & M32, ((e1 << 1) | (e0 >> 31)) & M32, ((e2 << 1) | (e1 >> 31)) & M32,
                ((e3 << 1) | (e2 >> 31)) & M32, ((e4 << 1) | (e3 >> 31)) & M32,
                (o1 << 1) & M32, ((o2 << 1) | (o1 >> 31)) & M32, ((o3 << 1) | (o2 >> 31)) & M32)

    def wide_reduce_t(self, canon, w):
        r = self._asm("wide_reduce_t", self._wenv(w))
        return self.fp_reduce160_t(canon, w[0], r["x1"], r["x2"], r["x3"], r["x4"])

    # ---- the hook's ops: the 16 output words of schnorr_b200_debug_fp_core for one item ----
    def op(self, name, args):
        if name.startswith("wide_"):
            w = tuple(args[0])
            if name == "wide_mac":
                w = self.wide_mac(w, args[1], args[2])
            elif name == "wide_mac_sqr":
                w = self.wide_mac_sqr(w, args[1])
            elif name == "wide_add64":
                w = self.wide_add64(w, args[1])
            elif name == "wide_double":
                w = self.wide_double(w)
            elif name == "wide_mac_loop":
                for _ in range(args[3]):
                    w = self.wide_mac(w, args[1], args[2])
            nc, cn = self.wide_reduce_t(False, w), self.wide_reduce_t(True, w)
            return list(w) + [lo(nc), hi(nc), lo(cn), hi(cn)] + [0] * 4
        f = {"reduce96_nc": self.fp_reduce96_nc, "reduce96": self.fp_reduce96,
             "reduce160_nc": lambda *x: self.fp_reduce160_t(False, *x),
             "reduce160": lambda *x: self.fp_reduce160_t(True, *x)}.get(name) or getattr(self, "fp_" + name)
        r = f(*args)
        return [lo(r), hi(r)] + [0] * 14
