"""Stan-subset front end: a Stan program + its data -> a fused value-and-gradient device function.

The reference hands ANY Stan program to BridgeStan (smcnuts/model/bridgestan.py:13-26: `StanModel(model_name,
model_path, data_path)` compiles it with stanc + Stan Math and evaluates log_density / log_density_gradient through
ctypes, one call per particle).  Here the program is translated into the C++ body of a model struct with the interface
of csrc/models.cuh (`eval(x, phi, A, B, g)`), which csrc/nuts_plugin.cuh instantiates into the same persistent NUTS
kernel and batched logp/grad kernel as the built-in models (SURVEY.md section 8 f3).  The same generated text also
compiles with plain g++ -- that is how the `not gpu` tests check it against the oracle densities.

What is generated
  * parameters on the unconstrained scale, Stan's transforms and log-Jacobians (lower -> lo + exp(u), upper,
    lower+upper -> scaled inverse logit; simplex, ordered and positive_ordered vectors through csrc/stan_transforms.cuh),
    declaration order = BridgeStan's unconstrained order.  The body sees one leaf per CONSTRAINED value (c[0 .. CDIM)) and
    accumulates its gradient over them; after the body one pullback per vector parameter maps it to the unconstrained
    coordinates and adds the gradient of its log-Jacobian (O(K) per vector, all Jacobians in A).  simplex is Stan's
    stick-breaking transform of releases up to 2.35 (what BridgeStan builds against those compute); later releases
    may use another simplex transform, which tests/test_bridgestan_pin.py would show.  The struct's static constrain(x, out)
    writes the CDIM constrained values with the same transform functions (smcb_model_constrain);
  * the split  logp(x, phi) = A(x) + phi * B(x): the data variable named `phi` is the tempering parameter
    (bridgestan.py:122-146 rewrites it in the data JSON); `target += phi * e` accumulates into B, everything else into A;
    all normalising constants of `target +=` statements are kept, `~` statements drop parameter-free terms (Stan's
    propto semantics under BridgeStan's defaults);
  * the gradient by statement-level forward-mode differentiation: every assignment's right-hand side is differentiated
    in reverse over its (small) expression DAG, and the adjoints of its leaves are pushed onto the sensitivities of the
    assigned variable -- only over the coordinates that variable can depend on;  loop-carried recurrences (arma's
    err[t-1]) therefore work, and loops stay loops (bounds are literals: scalar data is folded at generation time).

Supported subset (anything else raises StanSubsetError with the offending line):
  blocks functions (functions returning real, inlined at the call: no recursion, one return at the end) / data /
  transformed data / parameters / transformed parameters / model / generated quantities (below);  int, real, vector,
  row_vector, matrix (data and
  locals), array[..] (and the pre-2.33 `real y[N]` form);  lower/upper bounds on real parameters;  simplex[K], ordered[K],
  positive_ordered[K] (and arrays of them) as parameters, as data (validated at generation time: rows >= 0 summing to 1
  within 1e-8, strictly increasing) and as plain vectors in transformed parameters;  local declarations
  with initialisers, =, +=, -=, *=, /=, `target +=`, `~`, for and while loops, print (ignored), reject (the density becomes -inf, which is what the
  reference makes of a Stan exception), if / else (conditions on data, loop variables or
  parameter values; && || !), blocks;
  + - * / ^ .* ./, unary minus, indexing, exp log log1p sqrt fabs abs square inv inv_logit log1p_exp log_sum_exp(a, b)
  pow fmin fmax tanh sin cos lgamma (of data: tabulated at generation time; of parameters: differentiated with a digamma series);
  container-valued expressions: elementwise arithmetic and functions, matrix * vector, row_vector * vector,
  row_vector * matrix, sum mean dot_product dot_self rep_vector rep_row_vector rep_array, log_sum_exp(container) (max
  shifted; gradient = the softmax weights),
  whole-container assignment -- lowered onto element loops and accumulator locals of the scalar subset (`lower_stmt`);
  normal, std_normal, cauchy, student_t, double_exponential, logistic, lognormal, exponential, gamma, inv_gamma, weibull,
  beta, uniform densities; poisson, poisson_log, bernoulli, bernoulli_logit, binomial, binomial_logit, neg_binomial_2,
  neg_binomial_2_log mass functions --
  scalar or vectorised over container arguments and container-valued argument expressions;  dirichlet (alpha data or
  parameters), categorical (an int or int array outcome) and multinomial (an int array) of a vector argument, the integer
  outcomes being data known at generation time (tabulated into counts);
  matrices: cholesky_decompose(A) (symmetric within 1e-8 and positive definite, else the density is -inf), add_diag(A, d)
  (d real or vector), gp_exp_quad_cov(x, alpha, rho) (x array[] real or array[] vector), multi_normal_lpdf(y | mu, Sigma)
  and multi_normal_cholesky_lpdf(y | mu, L) (y and mu vectors or arrays of vectors; only the lower triangle of L is read,
  a diagonal entry <= 0 or not finite gives -inf; `~` drops -K/2 log 2 pi, and -sum log L_ii when the matrix depends on no
  parameter) -- lowered onto element loops of the scalar subset (`_Gen.mvn_terms`, `_Gen.cholesky_in_place`), the factor
  computed in place in the assigned matrix, loops with literal bounds kept rolled.  A covariance of multi_normal that is a
  data variable, and `matrix[K, K] L = cholesky_decompose(S);` in transformed data with S a data variable, are factored
  when the model is generated (numpy; not symmetric positive definite -> StanSubsetError with the line): an evaluation
  then only solves, O(K^2).
  Per-thread budget: the matrix locals of the density, values and tangents (8 bytes x entries x (1 + tangents an entry,
  the highest coordinate the matrix depends on + 1)), take at most _Gen.MAX_MATRIX_BYTES = 32 KiB; a program past it is
  refused with the line of the matrix that crosses it.  Local memory is reserved for every thread that can be resident
  (148 SMs x 2048 on a B200), so 32 KiB is about 10 GB of the device: the plug-in's NUTS kernel has a 34 KB stack frame
  at the budget (a 32-observation GP with 3 hyperparameters, profiles/gp_time.log).

Generated quantities (a separate output: `constrain()`, `param_names` and the density code do not change)
  a second struct `<struct_name>GQ` (GeneratedSource.gq_text) with generated_quantities(x, rng, out): value-only code
  (no sensitivities, no A / B split) of transformed data, transformed parameters and the block, over the constrained
  parameters; the outputs are the block's top-level int / real / vector / row_vector declarations and arrays of them
  (gq_names: BridgeStan's name.i.j, ints written as doubles).  Every construct of the model block is accepted, densities
  by value (`normal_lpdf(y[n] | mu[n], sigma)`), plus the _rng functions of csrc/stan_rng.cuh: normal, std_normal,
  student_t, cauchy, double_exponential, logistic, lognormal, exponential, gamma, inv_gamma, beta, uniform, bernoulli,
  bernoulli_logit, binomial, poisson, poisson_log, neg_binomial_2 (scalar, or vectorised into arrays) and categorical (of a
  vector), and multi_normal_rng(mu, Sigma) / multi_normal_cholesky_rng(mu, L) (a vector mean; K standard normals drawn
  in coordinate order, then mu + L z; into a vector or an element of an array of vectors; data covariances are factored
  per evaluation here).  `target +=`, `~`, phi and redeclared names are refused there, _rng calls everywhere else; G is at most
  MAX_GQ (one row of a particle block fits in shared memory).  A block outside this subset does
  not stop the model: its StanSubsetError text (with the line) is kept in GeneratedSource.gq_error and raised when gq
  values are requested.
"""
import json
import math
import re
from pathlib import Path


class StanSubsetError(NotImplementedError):
    pass


# Statement-level restructuring (a vectorised density fused into the loop that fills its vector, arrays reduced to rolling
# scalars).  tests/test_stan_fuzz.py switches it off to compare both forms of random programs; results must not change.
RESTRUCTURE = True


# ------------------------------------------------------------------------------------------------ tokenizer
_TOKEN = re.compile(r"""
    (?P<ws>\s+|//[^\n]*|\#[^\n]*|/\*.*?\*/)
  | (?P<str>"[^"\n]*")
  | (?P<num>(\d+\.\d*|\.\d+|\d+)([eE][+-]?\d+)?)
  | (?P<id>[A-Za-z_][A-Za-z_0-9]*)
  | (?P<op>\.\*|\./|\+=|-=|\*=|/=|<=|>=|==|!=|&&|\|\||[-+*/^()\[\]{},;:|<>=~'!])
""", re.X | re.S)


def _tokenize(text):
    toks, pos, line = [], 0, 1
    while pos < len(text):
        m = _TOKEN.match(text, pos)
        if not m:
            raise StanSubsetError(f"line {line}: cannot tokenize {text[pos:pos + 20]!r}")
        kind = m.lastgroup
        if kind != "ws":
            toks.append((kind, m.group(), line))
        line += m.group().count("\n")
        pos = m.end()
    toks.append(("eof", "", line))
    return toks


# ------------------------------------------------------------------------------------------------ parser (AST = tuples)
class _Parser:
    def __init__(self, text):
        self.t = _tokenize(text)
        self.i = 0
        self.orients = {}       # variable name -> "col" (vector) | "row" (row_vector) | "mat" (matrix): how `*` treats it
        self.ctypes = {}        # variable name -> "simplex" | "ordered" | "positive_ordered"
        self.gq_orients, self.gq_ctypes = {}, {}    # the same, with the declarations of generated quantities added

    def peek(self, k=0):
        return self.t[self.i + k]

    def next(self):
        tok = self.t[self.i]
        self.i += 1
        return tok

    def accept(self, val):
        if self.peek()[1] == val:
            return self.next()
        return None

    def expect(self, val):
        tok = self.next()
        if tok[1] != val:
            raise StanSubsetError(f"line {tok[2]}: expected {val!r}, found {tok[1]!r}")
        return tok

    def err(self, msg):
        raise StanSubsetError(f"line {self.peek()[2]}: {msg}")

    # ---- program
    def program(self):
        blocks = {}
        while self.peek()[0] != "eof":
            name = self.next()[1]
            if name in ("transformed", "generated"):
                name += " " + self.next()[1]
            self.expect("{")
            if name in ("data", "parameters"):
                blocks[name] = self.decls()
            elif name in ("model", "transformed data", "transformed parameters"):
                blocks[name] = self.stmts()
            elif name == "functions":
                blocks[name] = {}
                while self.peek()[1] != "}":
                    fname, fn = self.function()
                    blocks[name][fname] = fn
            elif name == "generated quantities":
                # parsed with orientations / vector kinds of its own (the density code must not see its declarations);
                # a block outside the subset is kept as its error: the density does not need it
                start, saved = self.i, (dict(self.orients), dict(self.ctypes))
                try:
                    blocks[name] = self.stmts()
                except StanSubsetError as e:
                    blocks["generated quantities error"] = str(e)
                    self.i = start
                    self.skip_block()
                    continue
                finally:
                    self.gq_orients, self.gq_ctypes = self.orients, self.ctypes
                    self.orients, self.ctypes = saved
            else:
                if not self.skip_block():
                    raise StanSubsetError(f"block {name!r} is outside the supported subset")
                continue
            self.expect("}")
        for need in ("parameters", "model"):
            if need not in blocks:
                raise StanSubsetError(f"missing block {need!r}")
        blocks.setdefault("data", [])
        return blocks

    def skip_block(self):
        """Skips to the `}` that closes the current block (consumed) -> whether the block was empty."""
        depth, empty = 1, True
        while depth:
            tok = self.next()
            depth += (tok[1] == "{") - (tok[1] == "}")
            empty = empty and tok[1] == "}"
            if tok[0] == "eof":
                self.err("unterminated block")
        return empty

    # ---- user-defined functions: name -> (return type, [(argument name, kind)], body statements, line);  kind is "int",
    #      "real" or "container" (vector / row_vector / array: bound by name at the call)
    def unsized_type(self):
        self.accept("data")
        dims = 0
        if self.accept("array"):
            self.expect("[")
            dims = 1
            while self.accept(","):
                dims += 1
            self.expect("]")
        base = self.next()[1]
        if base not in ("int", "real", "vector", "row_vector", "matrix", "void"):
            self.err(f"unsupported type {base!r} in a function signature")
        if self.accept("["):                  # pre-2.33: real[] x
            dims += 1
            while self.accept(","):
                dims += 1
            self.expect("]")
        return base, dims

    def function(self):
        line = self.peek()[2]
        rbase, rdims = self.unsized_type()
        name = self.next()
        if name[0] != "id":
            self.err("expected a function name")
        if rbase != "real" or rdims:
            raise StanSubsetError(f"line {line}: function {name[1]!r}: only functions returning real are supported")
        if name[1].endswith(("_lp", "_rng", "_lpdf", "_lpmf")):
            raise StanSubsetError(f"line {line}: function {name[1]!r}: _lp / _rng / _lpdf / _lpmf functions are outside the subset")
        self.expect("(")
        params = []
        while self.peek()[1] != ")":
            base, dims = self.unsized_type()
            arg = self.next()[1]
            if base == "matrix":
                raise StanSubsetError(f"line {line}: function {name[1]!r}: matrix arguments are outside the supported subset")
            params.append((arg, "container" if (dims or base in ("vector", "row_vector")) else base))
            self.accept(",")
        self.expect(")")
        self.expect("{")
        body = self.stmts()
        self.expect("}")
        return name[1], ("real", params, body, line)

    # ---- declarations: (name, base, shape[list of expr], lower, upper, init);  the constrained vector types are vectors
    #      whose kind is recorded in `ctypes` (name -> kind): enforced for parameters and data, plain vectors elsewhere
    _VECTOR_TYPES = ("simplex", "ordered", "positive_ordered")
    _REFUSED_TYPES = ("unit_vector", "sum_to_zero_vector", "sum_to_zero_matrix", "cholesky_factor_corr",
                      "cholesky_factor_cov", "cov_matrix", "corr_matrix", "column_stochastic_matrix",
                      "row_stochastic_matrix")
    _TYPES = ("int", "real", "vector", "row_vector", "array", "matrix") + _VECTOR_TYPES + _REFUSED_TYPES

    def is_decl(self):
        return self.peek()[1] in self._TYPES

    def bounds(self):
        lo = hi = None
        if self.accept("<"):
            while True:
                key = self.next()[1]
                self.expect("=")
                val = self.expr(no_gt=True)
                if key == "lower":
                    lo = val
                elif key == "upper":
                    hi = val
                else:
                    self.err(f"unsupported constraint {key!r}")
                if not self.accept(","):
                    break
            self.expect(">")
        return lo, hi

    def dims(self):
        out = []
        if self.accept("["):
            out.append(self.expr())
            while self.accept(","):
                out.append(self.expr())
            self.expect("]")
        return out

    def decl(self):
        line = self.peek()[2]
        shape = []
        base = self.next()[1]
        if base == "array":
            shape += self.dims()
            base = self.next()[1]
        if base in self._REFUSED_TYPES:
            raise StanSubsetError(f"line {line}: type {base!r} is outside the supported subset")
        ctype = None
        if base in self._VECTOR_TYPES:
            if self.peek()[1] == "<":
                raise StanSubsetError(f"line {line}: bounds on a {base} are outside the supported subset")
            ctype, base = base, "vector"
        lo, hi = self.bounds()
        orient = None
        if base in ("vector", "row_vector", "matrix"):
            orient = {"vector": "col", "row_vector": "row", "matrix": "mat"}[base]
            d = self.dims()
            if len(d) != (2 if base == "matrix" else 1):
                raise StanSubsetError(f"line {line}: {base} needs {2 if base == 'matrix' else 1} size(s)")
            shape += d
            base = "real"
        name = self.next()
        if name[0] != "id":
            raise StanSubsetError(f"line {line}: expected a variable name, found {name[1]!r}")
        if orient:
            self.orients[name[1]] = orient
        if ctype:
            self.ctypes[name[1]] = ctype
        shape += self.dims()          # pre-2.33 array syntax: real y[N]
        init = self.expr() if self.accept("=") else None
        self.expect(";")
        return (name[1], base, shape, lo, hi, init, line)

    def decls(self):
        out = []
        while self.peek()[1] != "}":
            out.append(self.decl())
        return out

    # ---- statements
    def stmts(self):
        out = []
        while self.peek()[1] != "}":
            out.append(self.stmt())
        return out

    def stmt(self):
        line = self.peek()[2]
        if self.is_decl():
            return ("decl", self.decl(), line)
        if self.accept("{"):
            body = self.stmts()
            self.expect("}")
            return ("block", body, line)
        if self.accept("for"):
            self.expect("(")
            var = self.next()[1]
            self.expect("in")
            lo = self.expr(no_colon=True)
            self.expect(":")
            hi = self.expr()
            self.expect(")")
            return ("for", var, lo, hi, [self.stmt()], line)
        if self.accept("if"):
            self.expect("(")
            cond = self.cond()
            self.expect(")")
            then = self.stmt()
            other = self.stmt() if self.accept("else") else None
            return ("if", cond, then, other, line)
        if self.accept("return"):
            e = self.expr()
            self.expect(";")
            return ("return", e, line)
        if self.accept("while"):
            self.expect("(")
            cond = self.cond()
            self.expect(")")
            return ("while", cond, self.stmt(), line)
        if self.peek()[1] in ("print", "reject") and self.peek(1)[1] == "(":
            what = self.next()[1]
            depth = 0
            while True:                       # the message (strings and expressions) is not evaluated
                tok = self.next()
                depth += (tok[1] == "(") - (tok[1] == ")")
                if tok[0] == "eof":
                    self.err(f"unterminated {what}")
                if depth == 0:
                    break
            self.expect(";")
            return (what, line)
        if self.peek()[1] in ("print", "reject"):
            raise StanSubsetError(f"line {line}: statement {self.peek()[1]!r} is outside the supported subset")
        if self.peek()[1] == "target" and self.peek(1)[1] == "+=":
            self.next(); self.next()
            e = self.expr()
            self.expect(";")
            return ("target", e, line)
        lhs = self.expr()
        if self.accept("~"):
            dist = self.next()[1]
            self.expect("(")
            args = [] if self.peek()[1] == ")" else [self.expr()]
            while self.accept(","):
                args.append(self.expr())
            self.expect(")")
            if self.peek()[1] == "T":
                raise StanSubsetError(f"line {line}: truncation T[,] is outside the supported subset")
            self.expect(";")
            return ("tilde", lhs, dist, args, line)
        op = self.next()[1]
        if op not in ("=", "+=", "-=", "*=", "/="):
            raise StanSubsetError(f"line {line}: expected an assignment, found {op!r}")
        rhs = self.expr()
        self.expect(";")
        return ("assign", lhs, op, rhs, line)

    # ---- conditions of `if`: || over && over ! over one comparison of two arithmetic expressions (or a bare expression)
    def cond(self):
        a = self.cond_and()
        while self.accept("||"):
            a = ("lor", a, self.cond_and())
        return a

    def cond_and(self):
        a = self.cond_not()
        while self.accept("&&"):
            a = ("land", a, self.cond_not())
        return a

    def cond_not(self):
        if self.accept("!"):
            return ("lnot", self.cond_not())
        if self.peek()[1] == "(":        # either a parenthesised condition or a parenthesised arithmetic operand
            save = self.i
            self.next()
            try:
                c = self.cond()
                self.expect(")")
                if self.peek()[1] in (")", "&&", "||") and c[0] in ("lor", "land", "lnot", "cmp"):
                    return c
            except StanSubsetError:
                pass
            self.i = save
        a = self.additive(False)
        if self.peek()[1] in ("<", ">", "<=", ">=", "==", "!="):
            op = self.next()[1]
            return ("cmp", op, a, self.additive(False))
        return ("cmp", "!=", a, ("num", 0.0, True))

    # ---- expressions
    def expr(self, no_gt=False, no_colon=False):
        return self.additive(no_gt)

    def additive(self, no_gt):
        a = self.multiplicative(no_gt)
        while self.peek()[1] in ("+", "-"):
            op = self.next()[1]
            a = ("bin", op, a, self.multiplicative(no_gt))
        return a

    def multiplicative(self, no_gt):
        a = self.unary(no_gt)
        while self.peek()[1] in ("*", "/", ".*", "./"):
            op = self.next()[1]
            a = ("bin", op, a, self.unary(no_gt))
        return a

    def unary(self, no_gt):
        if self.accept("-"):
            return ("neg", self.unary(no_gt))
        if self.accept("+"):
            return self.unary(no_gt)
        return self.power(no_gt)

    def power(self, no_gt):
        a = self.postfix()
        if self.accept("^"):
            return ("bin", "^", a, self.unary(no_gt))     # right associative, binds tighter than unary minus on its left
        return a

    def postfix(self):
        a = self.primary()
        while True:
            if self.peek()[1] == "[":
                a = ("idx", a, self.dims())
            elif self.peek()[1] == "'":
                self.err("transposition is outside the supported subset")
            else:
                return a

    def primary(self):
        tok = self.next()
        if tok[0] == "num":
            return ("num", float(tok[1]), "." not in tok[1] and "e" not in tok[1].lower())
        if tok[1] == "(":
            e = self.expr()
            self.expect(")")
            return e
        if tok[0] == "id":
            if self.peek()[1] == "(":
                self.next()
                args = []
                if self.peek()[1] != ")":
                    args.append(self.expr())
                    while self.accept(",") or self.accept("|"):
                        args.append(self.expr())
                self.expect(")")
                return ("call", tok[1], args, tok[2])
            return ("var", tok[1], tok[2])
        raise StanSubsetError(f"line {tok[2]}: unexpected {tok[1]!r}")


# ------------------------------------------------------------------------------------------------ expression DAG
class Node:
    """Real-valued expression node.  kind: const | param | local | data | ivar | un | bin.
    deps = frozenset of unconstrained coordinates the value can depend on."""
    __slots__ = ("kind", "op", "args", "val", "deps", "name", "idx")

    def __init__(self, kind, op=None, args=(), val=None, deps=frozenset(), name=None, idx=None):
        self.kind, self.op, self.args, self.val, self.deps, self.name, self.idx = kind, op, args, val, deps, name, idx


def _const(v):
    return Node("const", val=float(v))


def _is_const(n, v=None):
    return n.kind == "const" and (v is None or n.val == v)


def _un(op, a):
    if a.kind == "const":
        f = {"neg": lambda z: -z, "exp": math.exp, "log": lambda z: math.log(z) if z > 0 else (-math.inf if z == 0 else math.nan),
             "log1p": math.log1p, "sqrt": math.sqrt, "fabs": abs, "lgamma": math.lgamma, "tanh": math.tanh,
             "sin": math.sin, "cos": math.cos, "inv_logit": lambda z: 1.0 / (1.0 + math.exp(-z)),
             "log1p_exp": lambda z: max(z, 0.0) + math.log1p(math.exp(-abs(z)))}[op]
        return _const(f(a.val))
    return Node("un", op=op, args=(a,), deps=a.deps)


def _fold(op, x, y):
    try:
        if op == "+":
            return x + y
        if op == "-":
            return x - y
        if op == "*":
            return x * y
        if op == "/":
            return x / y if y != 0 else (math.nan if x == 0 else math.copysign(math.inf, x))
        if op in ("fmin", "fmax"):
            return min(x, y) if op == "fmin" else max(x, y)
        r = x ** y
        return r if isinstance(r, float) else math.nan
    except (OverflowError, ZeroDivisionError, ValueError):
        return math.nan


def _bin(op, a, b):
    if a.kind == "const" and b.kind == "const":
        return _const(_fold(op, a.val, b.val))
    if op == "+" and _is_const(a, 0.0):
        return b
    if op in "+-" and _is_const(b, 0.0):
        return a
    if op == "*" and (_is_const(a, 1.0)):
        return b
    if op in "*/" and _is_const(b, 1.0):
        return a
    if op == "^" and _is_const(b, 2.0):
        return Node("bin", op="*", args=(a, a), deps=a.deps)
    if op == "^" and _is_const(b, 1.0):
        return a
    return Node("bin", op=op, args=(a, b), deps=a.deps | b.deps)


def _add(*terms):
    out = terms[0]
    for t in terms[1:]:
        out = _bin("+", out, t)
    return out


def _sub(a, b):
    return _bin("-", a, b)


def _mul(a, b):
    return _bin("*", a, b)


def _div(a, b):
    return _bin("/", a, b)


def _log(a):
    return _un("log", a)


def _z(y, m, s):
    """(y - m) / s as a product with the reciprocal scale -- Stan Math's own arithmetic (inv_sigma), and the reciprocal
    of a parameter-only scale is computed once per evaluation instead of one division per observation"""
    return _mul(_sub(y, m), _div(_const(1.0), s))


_LOG_2PI, _LOG_PI = math.log(2.0 * math.pi), math.log(math.pi)

# log densities as sums of terms (each a Node): Stan's definitions with every normalising constant
_DENSITIES = {
    "normal": lambda y, m, s: [_const(-0.5 * _LOG_2PI), _un("neg", _log(s)), _mul(_const(-0.5), _bin("^", _z(y, m, s), _const(2.0)))],
    "cauchy": lambda y, m, s: [_const(-_LOG_PI), _un("neg", _log(s)), _un("neg", _un("log1p", _bin("^", _z(y, m, s), _const(2.0))))],
    "double_exponential": lambda y, m, s: [_const(-math.log(2.0)), _un("neg", _log(s)), _un("neg", _mul(_un("fabs", _sub(y, m)), _div(_const(1.0), s)))],
    "lognormal": lambda y, m, s: [_const(-0.5 * _LOG_2PI), _un("neg", _log(s)), _un("neg", _log(y)),
                                  _mul(_const(-0.5), _bin("^", _z(_log(y), m, s), _const(2.0)))],
    "student_t": lambda y, nu, m, s: [_sub(_un("lgamma", _mul(_const(0.5), _add(nu, _const(1.0)))), _un("lgamma", _mul(_const(0.5), nu))),
                                      _mul(_const(-0.5), _log(_mul(nu, _const(math.pi)))), _un("neg", _log(s)),
                                      _un("neg", _mul(_mul(_const(0.5), _add(nu, _const(1.0))),
                                                      _un("log1p", _div(_bin("^", _z(y, m, s), _const(2.0)), nu))))],
    "std_normal": lambda y: [_const(-0.5 * _LOG_2PI), _mul(_const(-0.5), _bin("^", y, _const(2.0)))],
    "logistic": lambda y, m, s: [_un("neg", _log(s)), _un("neg", _z(y, m, s)),
                                 _mul(_const(-2.0), _un("log1p_exp", _un("neg", _z(y, m, s))))],
    "weibull": lambda y, a, s: [_sub(_log(a), _log(s)), _mul(_sub(a, _const(1.0)), _sub(_log(y), _log(s))),
                                _un("neg", _bin("^", _div(y, s), a))],
    "binomial": lambda k, n, p: [_sub(_un("lgamma", _add(n, _const(1.0))),
                                      _add(_un("lgamma", _add(k, _const(1.0))), _un("lgamma", _add(_sub(n, k), _const(1.0))))),
                                 _mul(k, _log(p)), _mul(_sub(n, k), _un("log1p", _un("neg", p)))],
    "exponential": lambda y, b: [_log(b), _un("neg", _mul(b, y))],
    "gamma": lambda y, a, b: [_mul(a, _log(b)), _un("neg", _un("lgamma", a)), _mul(_sub(a, _const(1.0)), _log(y)), _un("neg", _mul(b, y))],
    "inv_gamma": lambda y, a, b: [_mul(a, _log(b)), _un("neg", _un("lgamma", a)), _un("neg", _mul(_add(a, _const(1.0)), _log(y))),
                                  _un("neg", _div(b, y))],
    "beta": lambda y, a, b: [_sub(_un("lgamma", _add(a, b)), _add(_un("lgamma", a), _un("lgamma", b))),
                             _mul(_sub(a, _const(1.0)), _log(y)), _mul(_sub(b, _const(1.0)), _un("log1p", _un("neg", y)))],
    "uniform": lambda y, a, b: [_un("neg", _log(_sub(b, a)))],
    "poisson": lambda k, lam: [_mul(k, _log(lam)), _un("neg", lam), _un("neg", _un("lgamma", _add(k, _const(1.0))))],
    "poisson_log": lambda k, eta: [_mul(k, eta), _un("neg", _un("exp", eta)), _un("neg", _un("lgamma", _add(k, _const(1.0))))],
    "neg_binomial_2": lambda k, mu, ph: [
        _sub(_un("lgamma", _add(k, ph)), _un("lgamma", ph)), _un("neg", _un("lgamma", _add(k, _const(1.0)))),
        _mul(k, _sub(_log(mu), _log(_add(mu, ph)))), _mul(ph, _sub(_log(ph), _log(_add(mu, ph))))],
    "neg_binomial_2_log": lambda k, eta, ph: [
        _sub(_un("lgamma", _add(k, ph)), _un("lgamma", ph)), _un("neg", _un("lgamma", _add(k, _const(1.0)))),
        _mul(k, _sub(eta, _add(eta, _un("log1p_exp", _sub(_log(ph), eta))))),
        _mul(ph, _sub(_log(ph), _add(eta, _un("log1p_exp", _sub(_log(ph), eta)))))],
    "bernoulli": lambda k, p: [_mul(k, _log(p)), _mul(_sub(_const(1.0), k), _un("log1p", _un("neg", p)))],
    "bernoulli_logit": lambda k, eta: [_mul(k, eta), _un("neg", _un("log1p_exp", eta))],
    "binomial_logit": lambda k, n, eta: [_sub(_un("lgamma", _add(n, _const(1.0))),
                                              _add(_un("lgamma", _add(k, _const(1.0))), _un("lgamma", _add(_sub(n, k), _const(1.0))))),
                                         _mul(k, eta), _un("neg", _mul(n, _un("log1p_exp", eta)))],
}
# densities of a whole vector argument (simplex-valued or counts), lowered by _Gen.vector_density
_VECTOR_DENSITIES = ("dirichlet", "categorical", "multinomial")
# multivariate normal densities of vectors (or arrays of them) under a covariance or its Cholesky factor (_Gen.mvn_terms)
_MVN_DENSITIES = ("multi_normal", "multi_normal_cholesky")
_MVN_RNGS = ("multi_normal_rng", "multi_normal_cholesky_rng")
# matrix functions lowered onto element loops; the loops with literal bounds of a statement that uses one stay rolled
# (`#pragma unroll 1`): fully unrolled, the O(N^3) nests of a factorisation multiply nvcc time, code size and spills
_MATRIX_FUNCS = ("cholesky_decompose", "add_diag", "gp_exp_quad_cov", "multi_normal_lpdf",
                 "multi_normal_cholesky_lpdf") + _MVN_RNGS
_DBL_MAX = 1.7976931348623157e308


def _calls_any(e, names):
    found = []
    _walk_exprs(e, lambda x: found.append(x) if x[0] == "call" and x[1] in names else None)
    return bool(found)


def _sum_exprs(terms, line):
    out = terms[0] if terms else ("num", 0.0, True)
    for t in terms[1:]:
        out = ("bin", "+", out, t)
    return out


# _rng functions of generated quantities (csrc/stan_rng.cuh) -> number of arguments
_RNG_ARITY = {"normal": 2, "std_normal": 0, "student_t": 3, "cauchy": 2, "double_exponential": 2, "logistic": 2,
              "lognormal": 2, "exponential": 1, "gamma": 2, "inv_gamma": 2, "beta": 2, "uniform": 2, "bernoulli": 1,
              "bernoulli_logit": 1, "binomial": 2, "poisson": 1, "poisson_log": 1, "neg_binomial_2": 2, "categorical": 1}


def _has_rng(e):
    found = []
    _walk_exprs(e, lambda x: found.append(x) if x[0] == "call" and str(x[1]).endswith("_rng") else None)
    return bool(found)


_UNARY_FUNCS = {"exp": "exp", "log": "log", "log1p": "log1p", "sqrt": "sqrt", "fabs": "fabs", "abs": "fabs", "lgamma": "lgamma",
                "tanh": "tanh", "sin": "sin", "cos": "cos", "inv_logit": "inv_logit", "log1p_exp": "log1p_exp"}


# ------------------------------------------------------------------------------------------------ scalar replacement
def _walk_exprs(e, fn):
    """fn(sub-expression) for every expression node under `e` (tuples whose first item is a node kind)"""
    if isinstance(e, tuple) and e and isinstance(e[0], str):
        fn(e)
        for x in e[1:]:
            _walk_exprs(x, fn)
    elif isinstance(e, (list, tuple)):
        for x in e:
            _walk_exprs(x, fn)


def _key(e):
    """Structural identity of an expression, source lines left out"""
    if isinstance(e, tuple) and e and isinstance(e[0], str):
        if e[0] == "var":
            return ("var", e[1])
        if e[0] == "call":
            return ("call", e[1], _key(e[2]))
        return tuple(_key(x) for x in e)
    if isinstance(e, (list, tuple)):
        return tuple(_key(x) for x in e)
    return e


def _flat(ss):
    """the statements of a list with plain blocks opened up (a block runs once, in order)"""
    out = []
    for st in ss:
        out += _flat(st[1]) if st[0] == "block" else [st]
    return out


def _assigned_names(ss, out):
    """names of all variables assigned anywhere under the statement list"""
    for st in ss:
        if st[0] == "assign":
            base = st[1] if st[1][0] == "var" else st[1][1]
            if base[0] == "var":
                out.add(base[1])
        elif st[0] == "block":
            _assigned_names(st[1], out)
        elif st[0] == "for":
            _assigned_names(st[4], out)
        elif st[0] == "while":
            _assigned_names([st[2]], out)
        elif st[0] == "if":
            _assigned_names([x for x in (st[2], st[3]) if x is not None], out)
        elif st[0] == "decl" and st[1][5] is not None:
            out.add(st[1][0])
    return out


def _demote_arrays(stmts):
    """Local arrays that are only ever read at the element written LAST (same index expression, no other element written
    in between, not across loop trips) -- `mu[n] = ...; y[n] ~ normal(mu[n], s);` inside a loop -- never need to be
    arrays: they become scalars, which keeps their values and sensitivities in registers instead of per-thread local
    memory (whole-series ARMA at N = 2^18: see profiles/r2_generated_models_*.log).  Returns the rewritten statements."""
    arrays, bad = {}, set()

    def find_decls(ss):
        for st in ss:
            if st[0] == "decl" and st[1][2]:
                name = st[1][0]
                if name in arrays or st[1][5] is not None:
                    bad.add(name)
                arrays[name] = st
            elif st[0] == "block":
                find_decls(st[1])
            elif st[0] == "for":
                find_decls(st[4])
            elif st[0] == "while":
                find_decls([st[2]])
            elif st[0] == "if":
                find_decls([x for x in (st[2], st[3]) if x is not None])
    find_decls(stmts)
    if not arrays:
        return stmts

    def reads(e, last):
        whole, indexed = [], []

        def visit(x):
            if x[0] == "idx" and x[1][0] == "var" and x[1][1] in arrays:
                indexed.append(id(x[1]))
                if last.get(x[1][1]) != _key(x[2]):      # the latest write went to another (or an unknown) element
                    bad.add(x[1][1])
            elif x[0] == "var" and x[1] in arrays:
                whole.append(x)
        _walk_exprs(e, visit)
        for x in whole:                                  # a bare name that is not the base of an index: whole-container use
            if id(x) not in indexed:
                bad.add(x[1])

    def written_in(ss, out):
        for st in ss:
            if st[0] == "assign":
                lhs = st[1]
                base = lhs if lhs[0] == "var" else lhs[1]
                if base[0] == "var" and base[1] in arrays:
                    out.add(base[1])
            elif st[0] == "block":
                written_in(st[1], out)
            elif st[0] == "for":
                written_in(st[4], out)
            elif st[0] == "while":
                written_in([st[2]], out)
            elif st[0] == "if":
                written_in([x for x in (st[2], st[3]) if x is not None], out)
        return out

    def child(ss, last, repeated, loop=None):
        """a statement list that runs conditionally or repeatedly: on entry of a repeated one the elements written inside
        hold whatever the previous trip left; on exit the parent no longer knows which element was written last.
        The one recurrence that is tracked: `for (t in lo:hi)` whose body writes V exactly once, unconditionally, at V[t],
        with V[lo - 1] the latest write before the loop -- then V[t - 1] is the latest write on entry of every trip."""
        inner = dict(last)
        touched = written_in(ss, set())
        if repeated:
            flat = _flat(ss)
            nested = written_in([st for st in flat if st[0] != "assign"], set())
            for v in touched:
                inner[v] = None
                tops = [st for st in flat if st[0] == "assign" and (st[1] if st[1][0] == "var" else st[1][1])[1:2] == (v,)]
                if (loop is not None and v not in nested and len(tops) == 1 and tops[0][1][0] == "idx" and tops[0][2] == "="
                        and _key(tops[0][1][2]) == (("var", loop[0]),) and loop[1][0] == "num"
                        and last.get(v) == (("num", loop[1][1] - 1.0, True),)):
                    inner[v] = (("bin", "-", ("var", loop[0]), ("num", 1.0, True)),)
        scan(ss, inner)
        for v in touched:
            last[v] = None

    def scan(ss, last):
        for st in ss:
            k = st[0]
            if k == "decl":
                if st[1][5] is not None:
                    reads(st[1][5], last)
            elif k == "block":
                scan(st[1], last)
            elif k == "for":
                reads((st[2], st[3]), last)
                child(st[4], last, True, loop=(st[1], st[2]))
            elif k == "while":
                for v in written_in([st[2]], set()):      # the condition of a later trip sees what the body wrote
                    last[v] = None
                reads(st[1], last)
                child([st[2]], last, True)
            elif k == "if":
                reads(st[1], last)
                child([st[2]], last, False)
                if st[3] is not None:
                    child([st[3]], last, False)
            elif k == "target":
                reads(st[1], last)
            elif k == "tilde":
                reads((st[1], st[3]), last)
            elif k == "assign":
                _, lhs, op, rhs, _ = st
                reads(rhs, last)
                if lhs[0] == "idx" and lhs[1][0] == "var" and lhs[1][1] in arrays:
                    reads(lhs[2], last)
                    if op != "=":
                        reads(lhs, last)
                    last[lhs[1][1]] = _key(lhs[2])
                else:
                    reads(lhs, last)          # a whole-container assignment (or a scalar): counts as a whole use
    scan(stmts, {})
    names = set(arrays) - bad
    if not names:
        return stmts

    def rewrite(e):
        if isinstance(e, tuple) and e and isinstance(e[0], str):
            if e[0] == "idx" and e[1][0] == "var" and e[1][1] in names:
                return e[1]
            if e[0] == "decl" and e[1][0] in names:
                d = e[1]
                return ("decl", (d[0], d[1], [], d[3], d[4], d[5], d[6]), e[2])
            return tuple(rewrite(x) for x in e)
        if isinstance(e, list):
            return [rewrite(x) for x in e]
        if isinstance(e, tuple):
            return tuple(rewrite(x) for x in e)
        return e
    return rewrite(stmts)


# ------------------------------------------------------------------------------------------------ lowering + emission
class _Var:
    """A data array, parameter or model-block local."""

    def __init__(self, name, kind, shape, base="real", offset=0, lower=None, upper=None, value=None, orient=None):
        self.name, self.kind, self.shape, self.base, self.offset = name, kind, shape, base, offset
        self.orient = orient         # "col" | "row" | "mat" | None (plain array): what `*` does with it
        self.lower, self.upper, self.value = lower, upper, value
        self.size = 1
        for s in shape:
            self.size *= s
        self.deps = frozenset()      # locals: coordinates the variable can depend on (fixpoint of the activity analysis)


class GeneratedSource:
    """Result of `generate`: C++ text of the model struct and what the host side needs to know about it."""

    def __init__(self, struct_name, text, dim, blob, param_names, transforms, digest, cdim, param_unc_names,
                 gq_text="", gq_names=(), gq_error=None):
        self.struct_name, self.text, self.dim, self.blob = struct_name, text, dim, blob
        self.param_names, self.transforms, self.digest = param_names, transforms, digest
        self.cdim, self.param_unc_names = cdim, param_unc_names      # constrained width, unconstrained names
        # generated quantities: the struct `<struct_name>GQ` (included after `text`), its output names in BridgeStan's
        # form, and -- for a block outside the subset -- the StanSubsetError text, raised when gq values are requested
        self.gq_text, self.gq_names, self.gq_error = gq_text, list(gq_names), gq_error
        self.gq_dim = len(self.gq_names)


class _Gen:
    MAX_DIM = 64
    MAX_GQ = 24576          # outputs of generated quantities: a row of a particle block fits in shared memory
    # matrix locals of one thread, values and tangents together (module docstring): every thread that can be resident
    # (148 SMs x 2048 on a B200) gets a stack frame of at least this much local memory, about 10 GB at 32 KiB
    MAX_MATRIX_BYTES = 32768

    def __init__(self, blocks, data, struct_name, orients=None, ctypes=None, value_only=False):
        self.blocks, self.struct_name = blocks, struct_name
        self.value_only = value_only    # generated quantities: values only (no sensitivities, no A / B split), _rng calls
        self.orients = orients or {}
        self.ctypes = ctypes or {}
        self.rolled = set()     # loop variables of matrix-function lowerings: emitted with `#pragma unroll 1`
        self.rolling = False    # while a statement that uses a matrix function is lowered: its fresh loops are rolled
        self.materialized = {}  # id(matrix-valued call) -> the local it is computed into (one statement's lowering)
        self.folded = {}        # data covariance name -> name of its Cholesky factor, computed at generation time
        self.decl_lines = {}    # local name -> line of its declaration
        self.lowered = {}       # id(statement) -> its scalar-subset replacement (list of statements) or None
        self.rng_stmts = {}     # id(statement) -> the statement with its draws ahead of it, or None (value-only mode)
        self.scopes = [set()]   # value-only mode: names declared in each enclosing scope (Stan refuses redeclarations)
        self.fresh = 0
        self.functions = blocks.get("functions", {})
        self.inline_depth = 0
        calls = {}
        for fname, fn in self.functions.items():
            found = set()
            _walk_exprs(fn[2], lambda x, found=found: found.add(x[1]) if x[0] == "call" and x[1] in self.functions else None)
            calls[fname] = found

        def reaches(a, b, seen):
            return any(c == b or (c not in seen and reaches(c, b, seen | {c})) for c in calls[a])
        for fname, fn in self.functions.items():
            if reaches(fname, fname, {fname}):
                raise StanSubsetError(f"line {fn[3]}: recursive function {fname!r} is outside the supported subset")
        self.decl_init = {}     # id(declaration with an initialiser) -> its assignment statement
        self.hoisted, self.prologue = {}, []   # expression text -> name of its once-per-evaluation constant; their definitions
        self.outer_pre = None   # while a statement is being lowered: where its loop-invariant scalar reductions go
        self.data_in = dict(data)
        self.vars = {}          # name -> _Var
        self.loop_vars = []     # stack of (name, c_name)
        self.blob = []
        self.lines = []
        self.indent = 2
        self.tmp = 0
        self.derived = {}       # (data array, shift) -> blob offset of its tabulated lgamma
        self.transforms = []    # per unconstrained coordinate: (kind, lo, hi) with kind in none/lower/upper/both or the
        #                         vector type (simplex / ordered / positive_ordered) the coordinate belongs to
        self.param_names = []   # constrained names, BridgeStan's form (theta.1 ... theta.K)
        self.param_unc_names = []
        self.blocks_of = []     # per parameter transform, in declaration order: (kind, lo, hi, unconstrained offset,
        #                         constrained offset, K) -- K = 1 for a scalar coordinate

    # ---- integer expressions (indices, bounds, sizes): folded to Python ints when no loop variable is involved
    def int_expr(self, e):
        """-> (int value or None, C text)"""
        k = e[0]
        if k == "num":
            if not e[2]:
                raise StanSubsetError(f"real literal {e[1]} where an integer is required")
            return int(e[1]), str(int(e[1]))
        if k == "var":
            for name, cname in reversed(self.loop_vars):
                if name == e[1]:
                    return None, cname
            v = self.vars.get(e[1])
            if v is not None and v.kind == "data" and v.base == "int" and not v.shape:
                return int(v.value), str(int(v.value))
            raise StanSubsetError(f"line {e[2]}: {e[1]!r} is not an integer constant or loop variable")
        if k == "neg":
            v, c = self.int_expr(e[1])
            return (None if v is None else -v), f"(-{c})"
        if k == "bin" and e[1] in "+-*/":
            (va, ca), (vb, cb) = self.int_expr(e[2]), self.int_expr(e[3])
            if va is not None and vb is not None:
                r = {"+": va + vb, "-": va - vb, "*": va * vb, "/": int(va / vb) if vb else 0}[e[1]]
                return r, str(r)
            return None, f"({ca} {e[1]} {cb})"
        if k == "idx":     # integer data array element used as an index is not supported (no use in the target programs)
            raise StanSubsetError("integer array elements as indices are outside the supported subset")
        raise StanSubsetError(f"unsupported integer expression {e!r}")

    def is_int_expr(self, e):
        try:
            self.int_expr(e)
            return True
        except StanSubsetError:
            return False

    # ---- flat 0-based element index of var[idx...] -> (int or None, C text)
    def flat_index(self, v, idx_exprs, line=0):
        if len(idx_exprs) != len(v.shape):
            raise StanSubsetError(f"line {line}: {v.name} has {len(v.shape)} dimension(s), indexed with {len(idx_exprs)}")
        val, text = 0, "0"
        for e, n in zip(idx_exprs, v.shape):
            iv, ic = self.int_expr(e)
            if iv is not None and not (1 <= iv <= n):
                raise StanSubsetError(f"line {line}: index {iv} of {v.name} is out of range 1..{n}")
            if val is not None and iv is not None:
                val = val * n + (iv - 1)
                text = str(val)
            else:
                text = f"(({text}) * {n} + ({ic}) - 1)"
                val = None
        return val, text

    # ---- real expressions -> Node
    def real(self, e):
        k = e[0]
        if k == "num":
            return _const(e[1])
        if k == "ideq":          # 1.0 where two integer expressions are equal, else 0.0 (the diagonal of add_diag)
            (va, ca), (vb, cb) = self.int_expr(e[1]), self.int_expr(e[2])
            if va is not None and vb is not None:
                return _const(1.0 if va == vb else 0.0)
            return Node("ivar", name=f"({ca} == {cb})")
        if k == "neg":
            return _un("neg", self.real(e[1]))
        if k == "bin":
            a, b = self.real(e[2]), self.real(e[3])
            return _bin(e[1], a, b)
        if k == "var" or k == "idx":
            base, idx = (e, []) if k == "var" else (e[1], e[2])
            if base[0] != "var":
                raise StanSubsetError("only named variables can be indexed")
            name = base[1]
            for lv, cname in reversed(self.loop_vars):
                if lv == name:
                    return Node("ivar", name=cname)
            v = self.vars.get(name)
            if v is None:
                raise StanSubsetError(f"line {base[2]}: unknown variable {name!r}")
            if name == "phi" and v.kind == "data":
                raise StanSubsetError(f"line {base[2]}: the tempering variable phi may only multiply a whole `target +=` term")
            if len(idx) < len(v.shape):
                raise StanSubsetError(f"line {base[2]}: whole-array use of {name!r} is only supported as a density argument")
            iv, ic = self.flat_index(v, idx, base[2])
            if v.kind == "data":
                if iv is not None:
                    return _const(v.value[iv] if v.shape else v.value)
                return Node("data", name=name, idx=f"{v.offset} + {ic}")
            if v.kind == "param":
                if iv is not None:
                    return Node("param", idx=str(v.offset + iv), val=v.offset + iv, deps=frozenset([v.offset + iv]))
                return Node("param", idx=f"{v.offset} + {ic}", val=None, deps=frozenset(range(v.offset, v.offset + v.size)))
            return Node("local", name=name, idx=(ic if v.shape else None), deps=v.deps)
        if k == "call":
            return self.call(e)
        raise StanSubsetError(f"unsupported expression {e!r}")

    def call(self, e):
        name, args, line = e[1], e[2], e[3]
        if name.endswith("_rng"):
            return self.rng_call(name, args, line)
        m = re.fullmatch(r"(\w+?)_(lpdf|lpmf|log)", name)
        if m and m.group(1) in _DENSITIES:
            return _add(*self.density_terms(m.group(1), args, line, vectorised=False))
        if name in _UNARY_FUNCS and len(args) == 1:
            return _un(_UNARY_FUNCS[name], self.real(args[0]))
        if name == "square" and len(args) == 1:
            return _bin("^", self.real(args[0]), _const(2.0))
        if name == "inv" and len(args) == 1:
            return _div(_const(1.0), self.real(args[0]))
        if name == "pow" and len(args) == 2:
            return _bin("^", self.real(args[0]), self.real(args[1]))
        if name in ("fmin", "fmax") and len(args) == 2:
            return _bin(name, self.real(args[0]), self.real(args[1]))
        if name == "log_sum_exp" and len(args) == 2:
            a, b = self.real(args[0]), self.real(args[1])
            return _add(a, _un("log1p_exp", _sub(b, a)))
        raise StanSubsetError(f"line {line}: function {name!r} is outside the supported subset")

    def rng_call(self, name, args, line):
        """One draw of a scalar _rng function (csrc/stan_rng.cuh); categorical_rng takes a whole vector variable."""
        if not self.value_only:
            raise StanSubsetError(f"line {line}: {name}: _rng functions are only allowed in generated quantities")
        dist = name[:-4]
        if dist not in _RNG_ARITY:
            raise StanSubsetError(f"line {line}: function {name!r} is outside the supported subset")
        if len(args) != _RNG_ARITY[dist]:
            raise StanSubsetError(f"line {line}: {name} takes {_RNG_ARITY[dist]} argument(s)")
        if dist == "categorical":
            v = self.vars.get(args[0][1]) if args[0][0] == "var" else None
            if v is None or len(v.shape) != 1:
                raise StanSubsetError(f"line {line}: categorical_rng takes a vector")
            ptr = {"data": f"&data[{v.offset}]", "param": f"&c[{v.offset}]"}.get(v.kind, f"v_{v.name}")
            return Node("rng", op=dist, name=ptr, idx=v.shape[0])
        return Node("rng", op=dist, args=tuple(self.real(a) for a in args))

    def density_terms(self, dist, args, line, vectorised=True):
        fn = _DENSITIES[dist]
        if len(args) != fn.__code__.co_argcount:
            raise StanSubsetError(f"line {line}: {dist} takes {fn.__code__.co_argcount} arguments")
        return [self.hoist_lgamma(t) for t in fn(*[self.real(a) for a in args])]

    def hoist_lgamma(self, n):
        """lgamma(data[i] + c) is tabulated at generation time as one more data array (the log-factorials of a count
        likelihood would otherwise be a run-time lgamma per observation and evaluation).  Generated quantities read the
        density's data blob as it is: there lgamma runs per evaluation."""
        if self.value_only:
            return n
        if n.kind not in ("un", "bin") or n.deps:
            if n.kind in ("un", "bin"):
                args = tuple(self.hoist_lgamma(a) for a in n.args)
                if any(x is not y for x, y in zip(args, n.args)):
                    return Node(n.kind, op=n.op, args=args, deps=n.deps)
            return n
        if n.kind == "un" and n.op == "lgamma":
            a, shift = n.args[0], 0.0
            if a.kind == "bin" and a.op in "+-" and a.args[0].kind == "data" and a.args[1].kind == "const":
                a, shift = a.args[0], (a.args[1].val if a.op == "+" else -a.args[1].val)
            if a.kind == "data":
                key = (a.name, shift)
                if key not in self.derived:
                    src = self.vars[a.name]
                    self.derived[key] = len(self.blob)
                    self.blob += [math.lgamma(z + shift) if z + shift > 0 else math.inf for z in src.value]
                off = self.derived[key] - self.vars[a.name].offset
                return Node("data", name=a.name, idx=f"{off} + {a.idx}")
            return n
        args = tuple(self.hoist_lgamma(a) for a in n.args)
        if any(x is not y for x, y in zip(args, n.args)):
            return Node(n.kind, op=n.op, args=args, deps=n.deps)
        return n

    # ---- whole-array arguments of a density: length of the broadcast, or None when every argument is scalar
    def vector_length(self, args):
        n = None
        for a in args:
            if a[0] == "var":
                v = self.vars.get(a[1])
                if v is not None and v.shape and not any(a[1] == lv for lv, _ in self.loop_vars):
                    if len(v.shape) != 1:
                        raise StanSubsetError(f"whole-array density argument {a[1]!r} must be one-dimensional")
                    if n is not None and n != v.shape[0]:
                        raise StanSubsetError(f"density arguments of different lengths ({n} and {v.shape[0]})")
                    n = v.shape[0]
        return n


    # ---- whole-container expressions: shapes, and their lowering onto the scalar subset ---------------------------------
    # A statement that uses vectors / matrices as values (elementwise arithmetic, matrix * vector, row_vector * vector,
    # sum / mean / dot_product / dot_self / rep_vector, densities of vector expressions) is rewritten into element loops
    # and accumulator locals of the scalar subset, which the differentiation machinery below already handles.
    _REDUCTIONS = ("sum", "mean", "dot_product", "dot_self")
    _REPS = ("rep_vector", "rep_row_vector", "rep_array")

    def is_loop_var(self, name):
        return any(name == lv for lv, _ in self.loop_vars)

    def shape(self, e):
        """-> (dims tuple, orientation of a 1-d result: "col" | "row" | None, or "mat")"""
        k = e[0]
        if k == "num" or k == "ideq":
            return (), None
        if k == "var" or k == "idx":
            base, idx = (e, []) if k == "var" else (e[1], e[2])
            if base[0] != "var":
                raise StanSubsetError("only named variables can be indexed")
            if self.is_loop_var(base[1]):
                return (), None
            v = self.vars.get(base[1])
            if v is None:
                raise StanSubsetError(f"line {base[2]}: unknown variable {base[1]!r}")
            rest = tuple(v.shape[len(idx):])
            if len(idx) > len(v.shape):
                raise StanSubsetError(f"line {base[2]}: {v.name} has {len(v.shape)} dimension(s), indexed with {len(idx)}")
            if not rest:
                return (), None
            if v.orient == "mat":
                return rest, ("mat" if len(rest) == 2 else "row")
            return rest, (v.orient if len(rest) == 1 else None)
        if k == "neg":
            return self.shape(e[1])
        if k == "bin":
            (da, oa), (db, ob) = self.shape(e[2]), self.shape(e[3])
            op = e[1]
            if not da:
                if db and op in ("/", "^"):
                    raise StanSubsetError(f"scalar {op} container is outside the supported subset (use ./ or a loop)")
                return db, ob
            if not db:
                return da, oa
            if op == "*":
                if oa == "mat" and ob == "col" and da[1] == db[0]:
                    return (da[0],), "col"
                if oa == "row" and ob == "col" and da == db:
                    return (), None
                if oa == "row" and ob == "mat" and da[0] == db[0]:
                    return (db[1],), "row"
                raise StanSubsetError("`*` between these containers is outside the supported subset (supported: matrix * vector, "
                                      "row_vector * vector, row_vector * matrix; elementwise products are `.*`)")
            if op in ("+", "-", ".*", "./"):
                if da != db:
                    raise StanSubsetError(f"operands of {op} have different sizes ({da} and {db})")
                return da, oa
            raise StanSubsetError(f"operator {op} between two containers is outside the supported subset")
        if k == "call":
            name, args = e[1], e[2]
            if (name in self._REDUCTIONS or name in self.functions or re.fullmatch(r"\w+_(lpdf|lpmf|log)", name)
                    or (name == "log_sum_exp" and len(args) == 1)):
                return (), None
            if name in self._REPS and len(args) == 2:
                n, _ = self.int_expr(args[1])
                if n is None:
                    raise StanSubsetError(f"line {e[3]}: the size of {name} must be a constant")
                return (n,), {"rep_vector": "col", "rep_row_vector": "row", "rep_array": None}[name]
            if name == "categorical_rng":
                return (), None
            if name in ("cholesky_decompose", "add_diag", "gp_exp_quad_cov") + _MVN_RNGS:
                return self.matrix_call_shape(name, args, e[3])
            shapes = [self.shape(a) for a in args]
            big = [sh for sh in shapes if sh[0]]
            if big and any(sh[0] != big[0][0] for sh in big):
                raise StanSubsetError(f"line {e[3]}: arguments of {name} have different sizes")
            if big and name.endswith("_rng"):       # vectorised draws are arrays, as in Stan
                return big[0][0], None
            return big[0] if big else ((), None)
        raise StanSubsetError(f"unsupported expression {e!r}")

    def fresh_name(self, prefix):
        self.fresh += 1
        name = f"{prefix}__{self.fresh}"       # Stan identifiers cannot end in two underscores: no collisions
        if self.rolling:
            self.rolled.add(name)
        return name

    def reduce(self, n, term_of, pre, line):
        """acc = sum over k = 1..n of term_of(k), emitted as scalar-subset statements appended to `pre` -> the accumulator"""
        acc, kv = self.fresh_name("r"), self.fresh_name("k")
        inner = []
        term = term_of(("var", kv, line), inner)
        body = inner + [("assign", ("var", acc, line), "+=", term, line)]
        pre.append(("decl", (acc, "real", [], None, None, ("num", 0.0, True), line), line))
        pre.append(("for", kv, ("num", 1.0, True), ("num", float(n), True), [("block", body, line)], line))
        return ("var", acc, line)

    def lower(self, e, ix, pre, line=0):
        """Scalar-subset expression for element `ix` (one index expression per dimension of shape(e)) of `e`.
        Statements the value needs first (accumulator loops) are appended to `pre`; those of a SCALAR sub-expression do
        not depend on the element, so they go to the statement level (`outer_pre`) and run once, before any element loop."""
        k = e[0]
        dims, orient = self.shape(e)
        if len(ix) != len(dims):
            raise StanSubsetError(f"line {line}: a container of {len(dims)} dimension(s) is used where {len(ix)} are expected")
        if not dims and self.outer_pre is not None:
            pre = self.outer_pre
        if k == "num" or k == "ideq":
            return e
        if k == "var":
            return ("idx", e, list(ix)) if ix else e
        if k == "idx":
            return ("idx", e[1], list(e[2]) + list(ix)) if ix else e
        if k == "neg":
            return ("neg", self.lower(e[1], ix, pre, line))
        if k == "bin":
            op, a, b = e[1], e[2], e[3]
            (da, oa), (db, ob) = self.shape(a), self.shape(b)
            if op == "*" and da and db:
                if oa == "mat" and ob == "col":      # (X v)[i] = sum_k X[i, k] v[k]
                    return self.reduce(da[1], lambda kk, p2: ("bin", "*", self.lower(a, [ix[0], kk], p2, line),
                                                               self.lower(b, [kk], p2, line)), pre, line)
                if oa == "row" and ob == "col":      # r * v = sum_k r[k] v[k]
                    return self.reduce(da[0], lambda kk, p2: ("bin", "*", self.lower(a, [kk], p2, line),
                                                               self.lower(b, [kk], p2, line)), pre, line)
                # row_vector * matrix: (r X)[j] = sum_k r[k] X[k, j]
                return self.reduce(da[0], lambda kk, p2: ("bin", "*", self.lower(a, [kk], p2, line),
                                                           self.lower(b, [kk, ix[0]], p2, line)), pre, line)
            return ("bin", op.lstrip("."), self.lower(a, ix if da else [], pre, line), self.lower(b, ix if db else [], pre, line))
        if k == "call":
            name, args, cl = e[1], e[2], e[3]
            if name in self._REPS and len(args) == 2:
                return self.lower(args[0], [], pre, cl)
            if name == "add_diag":
                i, j = ix
                d = args[1]
                dv = self.lower(d, [i] if self.shape(d)[0] else [], pre, cl)
                return ("bin", "+", self.lower(args[0], ix, pre, cl), ("bin", "*", ("ideq", i, j), dv))
            if name == "gp_exp_quad_cov":
                x, alpha, rho = args
                xd = self.shape(x)[0]
                if len(xd) == 1:
                    d2 = ("call", "square", [("bin", "-", self.lower(x, [ix[0]], pre, cl), self.lower(x, [ix[1]], pre, cl))], cl)
                else:
                    d2 = self.reduce(xd[1], lambda kk, p2: ("call", "square", [("bin", "-", self.lower(x, [ix[0], kk], p2, cl),
                                                                                  self.lower(x, [ix[1], kk], p2, cl))], cl), pre, cl)
                scale = ("bin", "/", ("num", -0.5, False), ("call", "square", [self.lower(rho, [], pre, cl)], cl))
                return ("bin", "*", ("call", "square", [self.lower(alpha, [], pre, cl)], cl),
                        ("call", "exp", [("bin", "*", d2, scale)], cl))
            if name == "cholesky_decompose" or name in _MVN_RNGS:
                return ("idx", self.materialize(e, pre, cl), list(ix))
            if name in self._REDUCTIONS:
                shapes = [self.shape(a)[0] for a in args]
                if len(args) != (2 if name == "dot_product" else 1) or any(len(d) != 1 for d in shapes) or len(set(shapes)) != 1:
                    raise StanSubsetError(f"line {cl}: {name} takes {'two' if name == 'dot_product' else 'one'} one-dimensional "
                                          f"container(s) of equal size")
                n = shapes[0][0]

                def term(kk, p2):
                    x = self.lower(args[0], [kk], p2, cl)
                    if name == "dot_product":
                        return ("bin", "*", x, self.lower(args[1], [kk], p2, cl))
                    return ("bin", "*", x, x) if name == "dot_self" else x
                total = self.reduce(n, term, pre, cl)
                return ("bin", "/", total, ("num", float(n), False)) if name == "mean" else total
            if name in self.functions:
                return self.lower(self.inline(name, args, pre, cl), [], pre, cl)
            if name == "categorical_rng" and len(args) == 1 and args[0][0] != "var":   # the vector is materialised first
                dims, orient = self.shape(args[0])
                if len(dims) != 1:
                    raise StanSubsetError(f"line {cl}: categorical_rng takes a vector")
                tmp = self.fresh_name("theta")
                self.vars[tmp] = _Var(tmp, "local", list(dims), "real", orient=orient)
                pre.append(("decl", (tmp, "real", [("num", float(dims[0]), True)], None, None, args[0], cl), cl))
                return ("call", name, [("var", tmp, cl)], cl)
            if name == "categorical_rng":
                return e
            if name == "log_sum_exp" and len(args) == 1:
                return self.log_sum_exp(args[0], pre, cl)
            m = re.fullmatch(r"(\w+?)_(lpdf|lpmf|log)", name)
            if m and m.group(1) in _VECTOR_DENSITIES:
                return _sum_exprs(self.vector_density(m.group(1), args, pre, cl), cl)
            if m and m.group(1) in _MVN_DENSITIES:
                return _sum_exprs(self.mvn_terms(m.group(1), args, pre, cl), cl)
            if m and m.group(1) in _DENSITIES:
                shapes = [self.shape(a)[0] for a in args]
                big = [d for d in shapes if d]
                if big:                               # a vectorised density inside a larger expression: sum over the elements
                    if any(len(d) != 1 or d != big[0] for d in big):
                        raise StanSubsetError(f"line {cl}: density arguments must be one-dimensional containers of equal size")
                    return self.reduce(big[0][0], lambda kk, p2: ("call", name, [self.lower(a, [kk] if d else [], p2, cl)
                                                                                 for a, d in zip(args, shapes)], cl), pre, cl)
                return ("call", name, [self.lower(a, [], pre, cl) for a in args], cl)
            return ("call", name, [self.lower(a, ix if self.shape(a)[0] else [], pre, cl) for a in args], cl)
        raise StanSubsetError(f"unsupported expression {e!r}")

    def one_dim(self, e, what, line):
        dims, _ = self.shape(e)
        if len(dims) != 1:
            raise StanSubsetError(f"line {line}: {what} takes a one-dimensional container")
        return dims[0]

    def log_sum_exp(self, v, pre, line):
        """log sum_k exp(v_k) = m + log sum_k exp(v_k - m) with m = max_k v_k; its gradient is the softmax weights (the
        derivatives through m cancel)"""
        n = self.one_dim(v, "log_sum_exp", line)
        mx, kv = self.fresh_name("m"), self.fresh_name("k")
        inner = []
        elem = self.lower(v, [("var", kv, line)], inner, line)
        pre.append(("decl", (mx, "real", [], None, None, self.lower(v, [("num", 1.0, True)], pre, line), line), line))
        pre.append(("for", kv, ("num", 2.0, True), ("num", float(n), True),
                    [("block", inner + [("assign", ("var", mx, line), "=", ("call", "fmax", [("var", mx, line), elem], line),
                                         line)], line)], line))
        total = self.reduce(n, lambda kk, p2: ("call", "exp", [("bin", "-", self.lower(v, [kk], p2, line), ("var", mx, line))],
                                               line), pre, line)
        return ("bin", "+", ("var", mx, line), ("call", "log", [total], line))

    def data_ints(self, e, what, line):
        """values of an integer data expression (a scalar, an array, or an element), known at generation time"""
        base, idx = (e, []) if e[0] == "var" else (e[1], e[2]) if e[0] == "idx" else (None, None)
        v = self.vars.get(base[1]) if base is not None and base[0] == "var" else None
        if v is None or v.kind != "data" or v.base != "int" or self.is_loop_var(base[1]):
            raise StanSubsetError(f"line {line}: the outcome of {what} must be integer data (an index known when the "
                                  f"model is generated)")
        if not v.shape:
            return [v.value]
        if len(idx) == len(v.shape):
            iv, _ = self.flat_index(v, idx, line)
            if iv is None:
                raise StanSubsetError(f"line {line}: the outcome of {what} must not depend on a loop variable")
            return [int(v.value[iv])]
        if idx:
            raise StanSubsetError(f"line {line}: the outcome of {what} must be a whole array or one element")
        return [int(z) for z in v.value]

    def vector_density(self, dist, args, pre, line):
        """dirichlet_lpdf(theta | alpha), categorical_lpmf(y | theta), multinomial_lpmf(y | theta) as scalar-subset
        expressions -> the list of its terms; with the integer outcomes tabulated into counts at generation time they
        all read sum_k c_k log theta_k plus normalising terms."""
        if len(args) != 2:
            raise StanSubsetError(f"line {line}: {dist} takes 2 arguments")

        def log_elem(e, k):
            return ("call", "log", [self.lower(e, [("num", float(k), True)], pre, line)], line)

        def weighted_logs(e, counts):
            terms = [("bin", "*", ("num", float(c), True), log_elem(e, k + 1)) for k, c in enumerate(counts) if c]
            return _sum_exprs(terms, line)

        if dist == "dirichlet":
            theta, alpha = args
            K = self.one_dim(theta, "dirichlet", line)
            if self.one_dim(alpha, "dirichlet", line) != K:
                raise StanSubsetError(f"line {line}: dirichlet arguments have different sizes")
            a = lambda kk: self.lower(alpha, [kk], pre, line)     # noqa: E731
            total = self.reduce(K, lambda kk, p2: self.lower(alpha, [kk], p2, line), pre, line)
            lg = self.reduce(K, lambda kk, p2: ("call", "lgamma", [self.lower(alpha, [kk], p2, line)], line), pre, line)
            body = []
            for k in range(1, K + 1):
                ak = a(("num", float(k), True))
                if not (ak[0] == "idx" and self.vars.get(ak[1][1]) is not None and self.vars[ak[1][1]].kind == "data"
                        and self.real(ak).kind == "const" and self.real(ak).val == 1.0):     # (1 - 1) log theta_k: no term
                    body.append(("bin", "*", ("bin", "-", ak, ("num", 1.0, True)), log_elem(theta, k)))
            body = _sum_exprs(body, line)
            return [("call", "lgamma", [total], line), ("neg", lg), body]
        y, theta = args
        K = self.one_dim(theta, dist, line)
        ys = self.data_ints(y, dist, line)
        if any(not (1 <= z <= K) for z in ys) and dist == "categorical":
            raise StanSubsetError(f"line {line}: categorical outcomes must lie in 1..{K}")
        if dist == "categorical":
            counts = [sum(1 for z in ys if z == k) for k in range(1, K + 1)]
            return [weighted_logs(theta, counts)]
        if len(ys) != K or any(z < 0 for z in ys):
            raise StanSubsetError(f"line {line}: multinomial counts must be {K} non-negative integers")
        norm = math.lgamma(sum(ys) + 1.0) - math.fsum(math.lgamma(z + 1.0) for z in ys)
        return [("num", norm, False), weighted_logs(theta, ys)]

    # ---- matrices: cholesky_decompose, add_diag, gp_exp_quad_cov, multi_normal(_cholesky) densities and draws -----------
    # All of them are lowered onto rolled element loops of the scalar subset, so that the tangents follow the existing
    # activity analysis (only the coordinates a matrix can depend on).  The factor is computed in place in the assigned
    # matrix; a covariance that is a data variable is factored when the model is generated (fold_cholesky).
    def square_dim(self, e, what, line):
        dims, orient = self.shape(e)
        if orient != "mat" or dims[0] != dims[1]:
            raise StanSubsetError(f"line {line}: {what} takes a square matrix (found a container of size {list(dims)})")
        return dims[0]

    def matrix_call_shape(self, name, args, line):
        arity = {"cholesky_decompose": 1, "add_diag": 2, "gp_exp_quad_cov": 3}.get(name, 2)
        if len(args) != arity:
            raise StanSubsetError(f"line {line}: {name} takes {arity} argument(s)")
        if name == "gp_exp_quad_cov":
            (dx, ox), ds = self.shape(args[0]), [self.shape(a)[0] for a in args[1:]]
            if ox is not None or len(dx) not in (1, 2) or any(ds):
                raise StanSubsetError(f"line {line}: gp_exp_quad_cov(x, alpha, rho) takes x as array[] real or array[] vector "
                                      f"and real alpha and rho")
            return (dx[0], dx[0]), "mat"
        if name in _MVN_RNGS:
            n = self.square_dim(args[1], name, line)
            dm, om = self.shape(args[0])
            if dm != (n,) or om not in ("col", "row"):
                raise StanSubsetError(f"line {line}: {name} takes a vector mean of size {n} (found a container of size "
                                      f"{list(dm)})")
            return (n,), "col"
        n = self.square_dim(args[0], name, line)
        if name == "add_diag" and self.shape(args[1])[0] not in ((), (n,)):
            raise StanSubsetError(f"line {line}: add_diag adds a real or a vector of size {n}")
        return (n, n), "mat"

    def loop(self, lo, hi, body_of, line):
        """`for (v in lo:hi) { body_of(v) }` with a fresh, rolled loop variable"""
        v = self.fresh_name("i")
        self.rolled.add(v)
        return ("for", v, lo, hi, [("block", body_of(("var", v, line)), line)], line)

    def local(self, dims, orient, line, init=None, prefix="t"):
        """a fresh local (declared now, so that the expressions built next can use it) and its declaration"""
        name = self.fresh_name(prefix)
        if orient:
            self.orients[name] = orient
        self.vars[name] = _Var(name, "local", list(dims), "real", orient=orient)
        return ("var", name, line), ("decl", (name, "real", [("num", float(d), True) for d in dims], None, None, init, line),
                                     line)

    def materialize(self, e, pre, line):
        """a matrix- or vector-valued call computed once, ahead of the statement, into a fresh local -> its name"""
        if id(e) not in self.materialized:
            dims, orient = self.shape(e)
            tmp, decl = self.local(dims, orient, line, prefix="m")
            out = self.outer_pre if self.outer_pre is not None else pre
            out.append(decl)
            out += self._lower_stmt_inner(("assign", tmp, "=", e, line), [])
            self.materialized[id(e)] = (e, tmp)
        return self.materialized[id(e)][1]

    def matrix_assign(self, lhs, rhs, line):
        """statements that assign cholesky_decompose(A) or a multi_normal(_cholesky)_rng draw to the whole container lhs"""
        name, args = rhs[1], rhs[2]
        one = ("num", 1.0, True)
        if name == "cholesky_decompose":
            n = self.square_dim(args[0], name, line)
            copy = self._lower_stmt_inner(("assign", lhs, "=", args[0], line), [])
            return copy + self.cholesky_in_place(lambda i, j: self.lower(lhs, [i, j], [], line), n, line)
        if not self.value_only:
            raise StanSubsetError(f"line {line}: {name}: _rng functions are only allowed in generated quantities")
        mu, S = args
        (n,), _ = self.shape(rhs)
        if name == "multi_normal_rng":
            S = self.materialize(("call", "cholesky_decompose", [S], line), [], line)
        elif S[0] not in ("var", "idx"):
            S = self.materialize(S, [], line)
        z, decl = self.local([n], "col", line, prefix="z")
        t = self.fresh_name("t")

        def mu_at(i, pre):
            return self.lower(mu, [i], pre, line)

        def finite(i):
            pre = []
            m = mu_at(i, pre)
            return pre + [("if", ("lnot", ("cmp", "<=", ("call", "fabs", [m], line), ("num", _DBL_MAX, False))),
                           ("reject", line), None, line)]

        def row(i):
            pre = []
            m = mu_at(i, pre)
            return pre + [("decl", (t, "real", [], None, None, m, line), line),
                          self.loop(one, i, lambda j: [("assign", ("var", t, line), "+=",
                                                        ("bin", "*", self.lower(S, [i, j], [], line), ("idx", z, [j])), line)],
                                    line),
                          ("assign", self.lower(lhs, [i], [], line), "=", ("var", t, line), line)]
        nn = ("num", float(n), True)
        # K standard normals in coordinate order, then mu + L z (Stan checks that mu is finite; the factor of Sigma, that
        # Sigma is symmetric positive definite)
        return [decl, self.loop(one, nn, lambda i: [("assign", ("idx", z, [i]), "=", ("call", "std_normal_rng", [], line),
                                                     line)], line),
                self.loop(one, nn, finite, line), self.loop(one, nn, row, line)]

    def cholesky_in_place(self, E, n, line):
        """Statements that replace the n x n matrix of elements E(i, j) (index expressions) by its lower Cholesky factor,
        column by column (each column reads the input's lower triangle and the finished columns only); then zero the
        upper triangle.  As Stan Math: the input is symmetric within 1e-8 (which NaN and infinite entries fail) and
        positive definite, or the density is -inf (reject)."""
        one, nn = ("num", 1.0, True), ("num", float(n), True)
        rej = ("reject", line)

        def minus1(v):
            return ("bin", "-", v, one)

        def not_le(a, b):
            return ("lnot", ("cmp", "<=", a, ("num", b, False)))
        check = self.loop(one, nn, lambda i: [self.loop(one, i, lambda j: [
            ("if", not_le(("call", "fabs", [("bin", "-", E(i, j), E(j, i))], line), 1e-8), rej, None, line)], line)], line)

        def column(j):
            s, t = self.fresh_name("s"), self.fresh_name("t")

            def row(i):
                return [("decl", (t, "real", [], None, None, E(i, j), line), line),
                        self.loop(one, minus1(j), lambda k: [("assign", ("var", t, line), "-=", ("bin", "*", E(i, k), E(j, k)),
                                                              line)], line),
                        ("assign", E(i, j), "=", ("bin", "/", ("var", t, line), E(j, j)), line)]
            return [("decl", (s, "real", [], None, None, E(j, j), line), line),
                    self.loop(one, minus1(j), lambda k: [("assign", ("var", s, line), "-=", ("call", "square", [E(j, k)], line),
                                                          line)], line),
                    ("if", ("lnot", ("cmp", ">", ("var", s, line), ("num", 0.0, False))), rej, None, line),
                    ("assign", E(j, j), "=", ("call", "sqrt", [("var", s, line)], line), line),
                    self.loop(("bin", "+", j, one), nn, row, line)]
        upper = self.loop(one, nn, lambda i: [self.loop(("bin", "+", i, one), nn, lambda j: [
            ("assign", E(i, j), "=", ("num", 0.0, True), line)], line)], line)
        return [check, self.loop(one, nn, column, line), upper]

    def cholesky_of_data(self, name, line):
        """Stan's cholesky_decompose of the data matrix `name`, now: the factor's values (row-major); a matrix that is not
        symmetric (within 1e-8) positive definite with finite entries is refused"""
        import numpy as np
        v = self.vars[name]
        n = v.shape[-1]
        a = np.array(v.value, dtype=np.float64).reshape(n, n)
        fac = None
        if np.all(np.isfinite(a)) and np.all(np.abs(a - a.T) <= 1e-8):
            try:
                fac = np.linalg.cholesky(a)
            except np.linalg.LinAlgError:
                pass
        if fac is None or not np.all(np.diag(fac) > 0.0):
            raise StanSubsetError(f"line {line}: data {name!r} is not a symmetric positive definite matrix")
        return [float(z) for z in fac.ravel()]

    def data_matrix(self, name, n, values):
        self.vars[name] = _Var(name, "data", [n, n], "real", offset=len(self.blob), value=values, orient="mat")
        self.orients[name] = "mat"
        self.blob += values

    def fold_cholesky(self, name, line):
        """the Cholesky factor of data covariance `name`, computed once at generation time into the data blob"""
        if name not in self.folded:
            values = self.cholesky_of_data(name, line)
            self.folded[name] = self.fresh_name(f"{name}_chol")
            self.data_matrix(self.folded[name], self.vars[name].shape[-1], values)
        return self.folded[name]

    def mvn_terms(self, dist, args, pre, line):
        """multi_normal(_cholesky)_lpdf(y | mu, S) -> its terms [-M K/2 log 2 pi, -M sum_i log L_ii, -1/2 sum_n |z_n|^2]
        with z_n = L^-1 (y_n - mu_n) by forward substitution (M vectors y_n / mu_n); the statements that compute the
        factor, log-determinant and quadratic form go to `pre`.  Under `~` the first term is always dropped and the second
        one when L depends on no parameter (ptarget)."""
        if len(args) != 3:
            raise StanSubsetError(f"line {line}: {dist} takes 3 arguments")
        y, mu, S = args
        K = self.square_dim(S, dist, line)

        def count(e, what):      # -> number of vectors of an array (None for one vector)
            d, o = self.shape(e)
            if len(d) == 1 and o in ("col", "row"):
                m, k = None, d[0]
            elif len(d) == 2 and o is None:
                m, k = d
            else:
                raise StanSubsetError(f"line {line}: {dist}: {what} must be a vector or an array of vectors")
            if k != K:
                raise StanSubsetError(f"line {line}: {dist}: {what} has {k} elements, the matrix is {K} x {K}")
            return m
        my, mm = count(y, "the outcome"), count(mu, "the location")
        if my is not None and mm is not None and my != mm:
            raise StanSubsetError(f"line {line}: {dist}: arrays of {my} outcomes and {mm} locations")
        M = my or mm or 1
        one, kk = ("num", 1.0, True), ("num", float(K), True)
        checked = False
        if dist == "multi_normal":
            if S[0] == "var" and self.vars[S[1]].kind == "data" and not self.value_only:
                S = ("var", self.fold_cholesky(S[1], line), line)
            else:
                S, checked = self.materialize(("call", "cholesky_decompose", [S], line), pre, line), True
        elif S[0] not in ("var", "idx"):
            S = self.materialize(S, pre, line)

        def E(i, j):
            return self.lower(S, [i, j], [], line)
        if S[0] == "var" and self.vars[S[1]].kind == "data":          # log-determinant of a data factor: folded now
            diag = [self.vars[S[1]].value[i * K + i] for i in range(K)]
            if all(0.0 < d < math.inf for d in diag):
                ld = ("num", math.fsum(math.log(d) for d in diag), False)
            else:
                pre.append(("reject", line))
                ld = ("num", 0.0, False)
        else:
            ld, decl = self.local([], None, line, ("num", 0.0, True), prefix="ld")
            pre.append(decl)
            dg = lambda i: E(i, i)           # noqa: E731

            def diag(i):
                bad = ("lor", ("lnot", ("cmp", ">", dg(i), ("num", 0.0, False))),
                       ("lnot", ("cmp", "<=", dg(i), ("num", _DBL_MAX, False))))
                return ([] if checked else [("if", bad, ("reject", line), None, line)]) + \
                    [("assign", ld, "+=", ("call", "log", [dg(i)], line), line)]
            pre.append(self.loop(one, kk, diag, line))
        q, qdecl = self.local([], None, line, ("num", 0.0, True), prefix="q")
        z, zdecl = self.local([K], "col", line, prefix="z")
        t = self.fresh_name("t")

        def solve(n):
            def row(i):
                inner = []
                yi = self.lower(y, [i] if my is None else [n, i], inner, line)
                mi = self.lower(mu, [i] if mm is None else [n, i], inner, line)
                return inner + [("decl", (t, "real", [], None, None, ("bin", "-", yi, mi), line), line),
                                self.loop(one, ("bin", "-", i, one), lambda j: [
                                    ("assign", ("var", t, line), "-=", ("bin", "*", E(i, j), ("idx", z, [j])), line)], line),
                                ("assign", ("idx", z, [i]), "=", ("bin", "/", ("var", t, line), E(i, i)), line),
                                ("assign", q, "+=", ("call", "square", [("idx", z, [i])], line), line)]
            return [self.loop(one, kk, row, line)]
        pre += [qdecl, zdecl]
        pre += [self.loop(one, ("num", float(M), True), solve, line)] if M > 1 else solve(None)
        return [("num", -0.5 * M * K * _LOG_2PI, False), ("neg", ("bin", "*", ("num", float(M), False), ld)),
                ("bin", "*", ("num", -0.5, False), q)]

    def is_plain(self, e):
        """Expressions the scalar machinery takes as they are: scalars without container operations inside, and whole
        one-dimensional variables (the vectorised density arguments of target_terms)."""
        dims, _ = self.shape(e)
        if dims:
            return e[0] == "var" and len(dims) == 1
        saved, self.outer_pre = self.outer_pre, []
        try:
            return self.lower(e, [], self.outer_pre) == e and not self.outer_pre
        finally:
            self.outer_pre = saved

    def element_loops(self, dims, body_of, line):
        """Nested `for` statements over a container of shape `dims`; body_of(index expressions) -> list of statements"""
        names = [self.fresh_name("i") for _ in dims]
        body = body_of([("var", nm, line) for nm in names])
        for nm, n in reversed(list(zip(names, dims))):
            body = [("for", nm, ("num", 1.0, True), ("num", float(n), True), [("block", body, line)], line)]
        return body

    def lower_stmt(self, s):
        key = id(s)
        if key not in self.lowered:
            self.lowered[key] = (s, self._lower_stmt(s))     # the statement is kept alive: ids are not reused
        return self.lowered[key][1]

    def _lower_stmt(self, s):
        self.outer_pre = []
        self.rolling = (s[0] == "tilde" and s[2] in _MVN_DENSITIES) or _calls_any(s, _MATRIX_FUNCS)
        self.materialized = {}
        try:
            out = self._lower_stmt_inner(s, self.outer_pre)
        finally:
            self.outer_pre = None
            self.rolling = False
        return out

    @staticmethod
    def _refs(e, name, out):
        """index lists of every use of variable `name` inside expression / statement tuples"""
        if isinstance(e, (tuple, list)):
            if len(e) >= 2 and e[0] == "idx" and isinstance(e[1], tuple) and e[1][:2] == ("var", name):
                out.append(list(e[2]))
                return out
            if len(e) >= 2 and e[0] == "var" and e[1] == name:
                out.append([])
                return out
            for x in e:
                _Gen._refs(x, name, out)
        return out

    def _lower_stmt_inner(self, s, pre):
        kind, line = s[0], s[-1]
        if kind == "target" or kind == "tilde":
            if kind == "target":
                tempered, e = self.scale_split(s[1])
                m = re.fullmatch(r"(\w+?)_(lpdf|lpmf|log)", e[1]) if e[0] == "call" else None
                dist, args = (m.group(1), e[2]) if (m and m.group(1) in _DENSITIES) else (None, None)
            else:
                tempered, dist, args = False, s[2], [s[1]] + s[3]
                if dist in _VECTOR_DENSITIES:       # propto: a term that depends on no parameter is dropped when emitted
                    return pre + [("ptarget", t, line) for t in self.vector_density(dist, args, pre, line)]
                if dist in _MVN_DENSITIES:
                    return pre + [("ptarget", t, line) for t in self.mvn_terms(dist, args, pre, line)]

            def rebuild(a):
                if kind == "tilde":
                    return ("tilde", a[0], dist, a[1:], line)
                call = ("call", e[1], a, e[3])
                return ("target", ("bin", "*", ("var", "phi", line), call) if tempered else call, line)
            if dist is not None:
                if all(self.is_plain(a) for a in args):
                    return None
                shapes = [self.shape(a)[0] for a in args]
                big = [d for d in shapes if d]
                if not big:
                    elems = [self.lower(a, [], pre, line) for a in args]
                    return pre + [rebuild(elems)]
                if any(len(d) != 1 or d != big[0] for d in big):
                    raise StanSubsetError(f"line {line}: density arguments must be one-dimensional containers of equal size")
                scalars = [None if d else self.lower(a, [], pre, line) for a, d in zip(args, shapes)]   # once, outside the loop

                def body(ix):
                    inner = []
                    elems = [self.lower(a, ix, inner, line) if d else sc for a, d, sc in zip(args, shapes, scalars)]
                    return inner + [rebuild(elems)]
                loops = self.element_loops(big[0], body, line)
                return pre + loops
            if kind == "tilde":
                return None
            e2 = self.lower(s[1], [], pre, line)
            return None if (e2 == s[1] and not pre) else pre + [("target", e2, line)]
        if kind == "assign":
            _, lhs, op, rhs, _ = s
            ldims, _ = self.shape(lhs)
            rdims, _ = self.shape(rhs)
            if op == "=" and rhs[0] == "call" and rhs[1] in ("cholesky_decompose",) + _MVN_RNGS:
                if rdims != ldims:
                    raise StanSubsetError(f"line {line}: assignment of a container of size {rdims} to one of size {ldims}")
                return pre + self.matrix_assign(lhs, rhs, line)
            if not ldims:
                r2 = self.lower(rhs, [], pre, line)
                return None if (r2 == rhs and not pre) else pre + [("assign", lhs, op, r2, line)]
            if rdims and rdims != ldims:
                raise StanSubsetError(f"line {line}: assignment of a container of size {rdims} to one of size {ldims}")
            name = (lhs if lhs[0] == "var" else lhs[1])[1]
            scalar_rhs = None if rdims else self.lower(rhs, [], pre, line)

            def body(ix):
                inner = []
                elem = self.lower(rhs, ix, inner, line) if rdims else scalar_rhs
                # Stan evaluates the right-hand side before it assigns: inside the element loop the assigned variable
                # may only be read at the element being written (reductions over it were hoisted ahead of the loop)
                own = self.lower(lhs, ix, inner, line)
                if any(r != own[2] for r in self._refs((inner, elem), name, [])):
                    raise StanSubsetError(f"line {line}: {name!r} is assigned from a product that reads its other elements; "
                                          f"assign to a second variable")
                return inner + [("assign", own, op, elem, line)]
            loops = self.element_loops(ldims, body, line)
            return pre + loops
        return None

    # ---- user-defined functions are inlined at the call ---------------------------------------------------------------
    def inline(self, name, args, pre, line):
        """Statements of the body (locals and loop variables renamed apart, arguments bound) appended to `pre`;
        -> the expression the function returns.  Integer arguments and plain names are substituted, other real arguments
        are evaluated once into a fresh local, container arguments must be variables (bound by name)."""
        rtype, params, body, fline = self.functions[name]
        if len(args) != len(params):
            raise StanSubsetError(f"line {line}: {name} takes {len(params)} argument(s)")
        if self.inline_depth >= 8:
            raise StanSubsetError(f"line {line}: recursive function {name!r} is outside the supported subset")
        if not body or body[-1][0] != "return":
            raise StanSubsetError(f"line {fline}: function {name!r} must end in its only return statement")
        env = {}
        for (pname, kind), a in zip(params, args):
            if kind == "container":
                if not self.shape(a)[0]:
                    raise StanSubsetError(f"line {line}: argument {pname!r} of {name} must be a container")
                if a[0] not in ("var", "idx"):      # a container expression: materialised into a fresh local first
                    dims, orient = self.shape(a)
                    if len(dims) != 1:
                        raise StanSubsetError(f"line {line}: argument {pname!r} of {name}: only one-dimensional expressions")
                    tmp = self.fresh_name(pname)
                    if orient:
                        self.orients[tmp] = orient
                    pre.append(("decl", (tmp, "real", [("num", float(dims[0]), True)], None, None, a, line), line))
                    a = ("var", tmp, line)
                env[pname] = a
            elif kind == "int" or a[0] in ("num", "var"):
                if kind == "int" and not self.is_int_expr(a):
                    raise StanSubsetError(f"line {line}: argument {pname!r} of {name} must be an integer constant expression")
                env[pname] = a
            else:
                tmp = self.fresh_name(pname)
                pre.append(("decl", (tmp, "real", [], None, None, a, line), line))
                env[pname] = ("var", tmp, line)

        def rename_decls(ss):
            for st in ss:
                if st[0] == "decl":
                    env[st[1][0]] = ("var", self.fresh_name(st[1][0]), st[2])
                    if st[1][0] in self.orients:
                        self.orients[env[st[1][0]][1]] = self.orients[st[1][0]]
                elif st[0] == "block":
                    rename_decls(st[1])
                elif st[0] == "for":
                    rename_decls(st[4])
                elif st[0] == "while":
                    rename_decls([st[2]])
                elif st[0] == "if":
                    rename_decls([x for x in (st[2], st[3]) if x is not None])
                elif st[0] == "return" and st is not body[-1]:
                    raise StanSubsetError(f"line {st[-1]}: function {name!r}: early returns are outside the supported subset")
                elif st[0] in ("target", "tilde"):
                    raise StanSubsetError(f"line {st[-1]}: function {name!r} must not touch the target")
        rename_decls(body)

        def sub(e, env):
            if isinstance(e, tuple) and e and isinstance(e[0], str):
                if e[0] == "var":
                    return env.get(e[1], e)
                if e[0] == "idx" and e[1][0] == "var" and e[1][1] in env:
                    base = env[e[1][1]]
                    idx = [sub(x, env) for x in e[2]]
                    if base[0] == "idx":             # the argument was a slice, x[n]: its indices come first
                        return ("idx", base[1], list(base[2]) + idx)
                    return ("idx", base, idx)
                if e[0] == "decl":
                    d = e[1]
                    return ("decl", (env[d[0]][1], d[1], [sub(x, env) for x in d[2]], None, None,
                                     None if d[5] is None else sub(d[5], env), d[6]), e[2])
                if e[0] == "for":
                    inner = dict(env)
                    inner[e[1]] = ("var", self.fresh_name(e[1]), e[5])
                    return ("for", inner[e[1]][1], sub(e[2], env), sub(e[3], env), sub(e[4], inner), e[5])
                if e[0] == "call":
                    return ("call", e[1], [sub(x, env) for x in e[2]], e[3])
                return tuple(sub(x, env) for x in e)
            if isinstance(e, list):
                return [sub(x, env) for x in e]
            return e
        def declare(ss):          # the returned expression is analysed before these statements are processed
            for st in ss:
                if st[0] == "decl":
                    nm, _, shp = st[1][0], st[1][1], st[1][2]
                    dims = [self.int_expr(d)[0] for d in shp]
                    if any(d is None for d in dims):
                        raise StanSubsetError(f"line {st[-1]}: local array sizes must be constants")
                    self.vars.setdefault(nm, _Var(nm, "local", dims, st[1][1], orient=self.orients.get(nm)))
                elif st[0] == "block":
                    declare(st[1])
                elif st[0] == "for":
                    self.loop_vars.append((st[1], st[1]))
                    declare(st[4])
                    self.loop_vars.pop()
                elif st[0] == "while":
                    declare([st[2]])
                elif st[0] == "if":
                    declare([x for x in (st[2], st[3]) if x is not None])
        self.inline_depth += 1
        try:
            new = sub(body[:-1], env)
            declare([x for x in pre if x[0] == "decl"])      # temporaries of the arguments
            declare(new)
            pre += new
            return sub(body[-1][1], env)
        finally:
            self.inline_depth -= 1

    # ---- a vectorised density over a local vector, moved to where the elements are produced ---------------------------
    def fuse_vector_densities(self, stmts):
        """`for (t in 2:T) { ...; err[t] = ...; }  target += phi * normal_lpdf(err | 0, sigma);` (the Stan manual's ARMA and
        most time-series programs) stores the whole series and its sensitivities per thread only to read them back once.
        When every element of the vector is written exactly once -- by constant-index assignments and by ONE loop that
        assigns V[t] unconditionally -- and the other density arguments involve no model-block local, the density
        statement is applied element by element right after each write instead; the array then usually reduces to a
        scalar (_demote_arrays).  Only the order in which terms are added to the accumulators changes."""
        stmts = list(stmts)
        locals_ = {}
        for st in stmts:
            if st[0] == "decl":
                locals_[st[1][0]] = st
        all_locals = set()

        def collect(ss):
            for st in ss:
                if st[0] == "decl":
                    all_locals.add(st[1][0])
                elif st[0] == "block":
                    collect(st[1])
                elif st[0] == "for":
                    collect(st[4])
                elif st[0] == "while":
                    collect([st[2]])
                elif st[0] == "if":
                    collect([x for x in (st[2], st[3]) if x is not None])
        collect(stmts)
        m = 0
        while m < len(stmts):
            fused = self._fuse_one(stmts, m, locals_, all_locals)
            if fused is None:
                m += 1
            else:
                stmts = fused
                m = 0
        return stmts

    def _fuse_one(self, stmts, m, locals_, all_locals):
        st = stmts[m]
        line = st[-1]
        if st[0] == "target":
            tempered, e = self.scale_split(st[1])
            mm = re.fullmatch(r"(\w+?)_(lpdf|lpmf|log)", e[1]) if e[0] == "call" else None
            if not (mm and mm.group(1) in _DENSITIES):
                return None
            args = list(e[2])
        elif st[0] == "tilde" and st[2] in _DENSITIES:
            args = [st[1]] + list(st[3])
        else:
            return None
        whole = [a for a in args if a[0] == "var" and a[1] in locals_ and len(locals_[a[1]][1][2]) == 1
                 and locals_[a[1]][1][5] is None]
        if len(whole) != 1:
            return None
        V = whole[0][1]
        n = self.int_expr(locals_[V][1][2][0])[0]
        if n is None:
            return None
        kinds = []           # per argument: "V", "container" (whole data / parameter vector: indexed too) or "scalar"
        for a in args:
            if a is whole[0]:
                kinds.append("V")
                continue
            names = []
            _walk_exprs(a, lambda x: names.append(x[1]) if x[0] == "var" else None)
            if any(nm in all_locals for nm in names):
                return None
            v = self.vars.get(a[1]) if a[0] == "var" else None
            if v is not None and v.shape:
                if v.shape != [n]:
                    return None
                kinds.append("container")
            else:
                try:
                    if self.shape(a)[0]:
                        return None          # container-valued expression: left to the lowering pass
                except StanSubsetError:
                    return None
                kinds.append("scalar")

        def element(ix):
            a2 = [("idx", a, [ix]) if k != "scalar" else a for a, k in zip(args, kinds)]
            if st[0] == "tilde":
                return ("tilde", a2[0], st[2], a2[1:], line)
            call = ("call", e[1], a2, e[3])
            return ("target", ("bin", "*", ("var", "phi", line), call) if tempered else call, line)
        # the writes of V ahead of the statement
        covered, out, loops = [], [], 0
        for j, sj in enumerate(stmts[:m]):
            if V not in _assigned_names([sj], set()):
                out.append(sj)
                continue
            if (sj[0] == "assign" and sj[2] == "=" and sj[1][0] == "idx" and len(sj[1][2]) == 1 and sj[1][2][0][0] == "num"
                    and sj[1][2][0][2]):
                c = int(sj[1][2][0][1])
                covered.append(c)
                out += [sj, element(("num", float(c), True))]
                continue
            if sj[0] != "for":
                return None
            lo, hi = self.int_expr(sj[2])[0], self.int_expr(sj[3])[0]
            if lo is None or hi is None or loops:
                return None
            loops += 1
            flat = _flat(sj[4])
            tops = [x for x in flat if x[0] == "assign" and (x[1] if x[1][0] == "var" else x[1][1])[1:2] == (V,)]
            if (len(tops) != 1 or V in _assigned_names([x for x in flat if x[0] != "assign"], set()) or tops[0][2] != "="
                    or tops[0][1][0] != "idx" or _key(tops[0][1][2]) != (("var", sj[1]),)):
                return None
            covered += list(range(lo, hi + 1))

            def with_element(ss):
                res = []
                for x in ss:
                    if x is tops[0]:
                        res += [x, element(("var", sj[1], line))]
                    elif x[0] == "block":
                        res.append(("block", with_element(x[1]), x[2]))
                    else:
                        res.append(x)
                return res
            out.append(("for", sj[1], sj[2], sj[3], with_element(sj[4]), sj[5]))
        if sorted(covered) != list(range(1, n + 1)):
            return None
        return out + stmts[m + 1:]

    # ---- conditions of `if`
    def cond_text(self, c, line):
        if c[0] in ("lor", "land"):
            return f"({self.cond_text(c[1], line)} {'||' if c[0] == 'lor' else '&&'} {self.cond_text(c[2], line)})"
        if c[0] == "lnot":
            return f"(!{self.cond_text(c[1], line)})"
        sides = []
        for e in (c[2], c[3]):
            if self.is_int_expr(e):
                sides.append(self.int_expr(e)[1])
            else:
                pre = []
                e2 = self.lower(e, [], pre, line)
                if pre:
                    raise StanSubsetError(f"line {line}: container operations inside a condition are outside the supported subset")
                if self.shape(e)[0]:
                    raise StanSubsetError(f"line {line}: a condition compares scalars")
                sides.append(self.emit_value_and_adjoints(self.real(e2))[0])
        return f"({sides[0]} {c[1]} {sides[1]})"

    # ---- emission helpers
    def emit(self, text):
        self.lines.append("    " * self.indent + text)

    def hoist(self, text):
        """Name of the once-per-evaluation constant `text` (an expression of parameters and literals only)."""
        nm = self.hoisted.get(text)
        if nm is None:
            nm = self.hoisted[text] = f"h{len(self.hoisted) + 1}"
            self.prologue.append(f"const double {nm} = {text};")
        return nm

    def new_tmp(self, prefix="t"):
        self.tmp += 1
        return f"{prefix}{self.tmp}"

    @staticmethod
    def lit(v):
        if v != v:
            return "NAN"
        if v in (math.inf, -math.inf):
            return "INFINITY" if v > 0 else "(-INFINITY)"
        r = repr(float(v))
        return f"({r})" if r.startswith("-") else r

    def topo(self, root):
        order, seen = [], set()

        def visit(n):
            if id(n) in seen:
                return
            seen.add(id(n))
            for a in n.args:
                visit(a)
            order.append(n)
        visit(root)
        return order

    def emit_value_and_adjoints(self, root):
        """Straight-line code for the value of `root` and the adjoints of its differentiable leaves.
        -> (value C name, [(leaf node, adjoint C text)])"""
        order = self.topo(root)
        name = {}
        fixed = {}       # nodes built from constants and parameters at constant indices only: the same value throughout one
        #                  evaluation, so they are computed once in the prologue of eval() and shared (log(sigma), 1 / sigma ...)
        for n in order:
            fixed[id(n)] = (n.kind == "const" or (n.kind == "param" and n.val is not None)
                            or (n.kind in ("un", "bin") and all(fixed[id(a)] for a in n.args)))
            if n.kind == "const":
                name[id(n)] = self.lit(n.val)
            elif n.kind == "param":
                name[id(n)] = f"c[{n.idx}]"
            elif n.kind == "local":
                name[id(n)] = f"v_{n.name}" + (f"[{n.idx}]" if n.idx is not None else "")
            elif n.kind == "data":
                name[id(n)] = f"data[{n.idx}]"
            elif n.kind == "ivar":
                name[id(n)] = f"(double){n.name}"
            elif n.kind == "rng":       # a draw: never shared between evaluations, never hoisted
                a = [name[id(x)] for x in n.args] + ["rng"]
                fn = f"categorical_rng<{n.idx}>" if n.op == "categorical" else f"{n.op}_rng"
                t = self.new_tmp()
                self.emit(f"const double {t} = smcb::stan::{fn}({n.name + ', ' if n.op == 'categorical' else ''}"
                          f"{', '.join(a)});")
                name[id(n)] = t
            else:
                a = [name[id(x)] for x in n.args]
                if n.kind == "un":
                    text = {"neg": f"-{a[0]}", "inv_logit": f"smcgen_inv_logit({a[0]})", "log1p_exp": f"smcgen_log1p_exp({a[0]})",
                            "exp": f"smcb::fast_exp({a[0]})"}.get(
                        n.op, f"{n.op}({a[0]})")
                elif n.op == "^":
                    text = f"sqrt({a[0]})" if _is_const(n.args[1], 0.5) else f"pow({a[0]}, {a[1]})"
                elif n.op in ("fmin", "fmax"):
                    text = f"{n.op}({a[0]}, {a[1]})"
                else:
                    text = f"{a[0]} {n.op} {a[1]}"
                if fixed[id(n)]:
                    name[id(n)] = self.hoist(text)
                    continue
                t = self.new_tmp()
                self.emit(f"const double {t} = {text};")
                name[id(n)] = t
        if self.value_only:
            return name[id(root)], []
        # reverse sweep over the nodes that depend on parameters
        adj = {id(root): ["1.0"]}
        leaves = []
        for n in reversed(order):
            if not n.deps or id(n) not in adj:
                continue
            terms = adj[id(n)]
            a_text = terms[0] if len(terms) == 1 else "(" + " + ".join(terms) + ")"
            if n.kind in ("param", "local"):
                leaves.append((n, a_text))
                continue
            if len(terms) > 1 or len(a_text) > 24:
                t = self.new_tmp("a")
                self.emit(f"const double {t} = {a_text};")
                a_text = t
            v = name[id(n)]
            xs = [name[id(x)] for x in n.args]

            def recip(k):
                return self.hoist(f"1.0 / {xs[k]}") if fixed[id(n.args[k])] else f"(1.0 / {xs[k]})"

            def push(child, factor):
                if child.deps:
                    term = a_text if factor is None else factor if a_text == "1.0" else f"{a_text} * {factor}"
                    adj.setdefault(id(child), []).append(term)
            if n.kind == "un":
                x = xs[0]
                push(n.args[0], recip(0) if n.op == "log" else
                     {"neg": "(-1.0)", "exp": v, "log1p": f"(1.0 / (1.0 + {x}))",
                                 "sqrt": f"(0.5 / {v})", "fabs": f"copysign(1.0, {x})", "tanh": f"(1.0 - {v} * {v})",
                                 "sin": f"cos({x})", "cos": f"(-sin({x}))", "inv_logit": f"({v} * (1.0 - {v}))",
                                 "lgamma": f"smcgen_digamma({x})",
                                 "log1p_exp": f"smcgen_inv_logit({x})"}[n.op])
            elif n.op == "+":
                push(n.args[0], None); push(n.args[1], None)
            elif n.op == "-":
                push(n.args[0], None); push(n.args[1], "(-1.0)")
            elif n.op == "*":
                if n.args[0] is n.args[1]:
                    push(n.args[0], f"(2.0 * {xs[0]})")          # a square (`^ 2` is built as x * x)
                else:
                    push(n.args[0], xs[1]); push(n.args[1], xs[0])
            elif n.op == "/":
                push(n.args[0], recip(1)); push(n.args[1], f"(-{v} * {recip(1)})")
            elif n.op in ("fmin", "fmax"):       # the gradient follows the selected argument (the first one on ties)
                first = f"({xs[0]} {'<=' if n.op == 'fmin' else '>='} {xs[1]})"
                push(n.args[0], f"({first} ? 1.0 : 0.0)"); push(n.args[1], f"({first} ? 0.0 : 1.0)")
            elif n.op == "^":
                if _is_const(n.args[1], 0.5):
                    push(n.args[0], f"(0.5 / {v})")
                else:
                    push(n.args[0], f"({xs[1]} * pow({xs[0]}, {xs[1]} - 1.0))")
                    push(n.args[1], f"({v} * log({xs[0]}))")
        return name[id(root)], leaves

    def emit_sensitivities(self, target_of, leaves, deps, accumulate):
        """d_target[k] (+)= sum over the leaves of adjoint * d leaf / d x_k, coordinate by coordinate.
        target_of(k) -> C lvalue of coordinate k;  param leaves with a run-time index scatter through `dyn`."""
        per_k = {k: [] for k in sorted(deps)}
        dynamic = []
        for n, a in leaves:
            if n.kind == "param":
                if n.val is not None:
                    per_k[n.val].append(f"{a} * dc[{n.val}]")
                else:
                    dynamic.append((n, a))
            else:
                vd = f"d_{n.name}" + (f"[{n.idx}]" if n.idx is not None else "")
                for k in sorted(n.deps):
                    per_k[k].append(f"{a} * {vd}[{k}]")
        for k in sorted(deps):
            terms = per_k[k]
            if accumulate:
                if terms:
                    self.emit(f"{target_of(k)} += {' + '.join(terms)};")
            else:
                self.emit(f"{target_of(k)} = {' + '.join(terms) if terms else '0.0'};")
        for n, a in dynamic:
            self.emit(f"{target_of(n.idx)} += {a} * dc[{n.idx}];")

    # ---- statements
    def scale_split(self, e):
        """`phi * E` (phi anywhere among the top-level factors) -> (True, E); otherwise (False, e)."""
        def strip(x):
            if x[0] == "var" and x[1] == "phi" and self.vars.get("phi") is not None and self.vars["phi"].kind == "data":
                return True, None
            if x[0] == "bin" and x[1] == "*":
                fa, ra = strip(x[2])
                if fa:
                    return True, x[3] if ra is None else ("bin", "*", ra, x[3])
                fb, rb = strip(x[3])
                if fb:
                    return True, x[2] if rb is None else ("bin", "*", x[2], rb)
            return False, x
        found, rest = strip(e)
        if found and rest is None:
            rest = ("num", 1.0, True)
        return found, rest

    def target_terms(self, e, line, drop_constant_terms):
        """Emit `target += e` (possibly a vectorised density) into the A or B accumulators."""
        tempered, e = self.scale_split(e)
        acc = "B" if tempered else "A"
        vec_n, m = None, None
        if e[0] == "call":
            m = re.fullmatch(r"(\w+?)_(lpdf|lpmf|log)", e[1])
            m = m if (m and m.group(1) in _DENSITIES) else None
            if m:
                vec_n = self.vector_length(e[2])
        if vec_n is not None:     # vectorised density: an element loop with scalar arguments broadcast
            cname = self.new_tmp("i")
            if vec_n <= 16:
                self.emit("#pragma unroll")
            self.emit(f"for (int {cname} = 1; {cname} <= {vec_n}; ++{cname}) {{")
            self.indent += 1
            self.loop_vars.append((cname, cname))
            args = [("idx", a, [("var", cname, line)]) if (a[0] == "var" and self.vars.get(a[1]) is not None and self.vars[a[1]].shape
                                                          and not any(a[1] == lv for lv, _ in self.loop_vars[:-1])) else a for a in e[2]]
            self.add_to_target(_add(*self.filter_terms(self.density_terms(m.group(1), args, line), drop_constant_terms)), acc)
            self.loop_vars.pop()
            self.indent -= 1
            self.emit("}")
            return
        node = _add(*self.filter_terms(self.density_terms(m.group(1), e[2], line), drop_constant_terms)) if m else self.real(e)
        if drop_constant_terms and not node.deps:
            return
        self.add_to_target(node, acc)

    @staticmethod
    def filter_terms(terms, drop_constant_terms):
        kept = [t for t in terms if t.deps] if drop_constant_terms else list(terms)
        return kept or [_const(0.0)]

    def add_to_target(self, node, acc):
        self.emit("{")
        self.indent += 1
        val, leaves = self.emit_value_and_adjoints(node)
        self.emit(f"{acc} += {val};")
        self.emit_sensitivities(lambda k: f"g{acc}[{k}]", leaves, node.deps, accumulate=True)
        self.indent -= 1
        self.emit("}")

    def assign(self, lhs, op, rhs_node, line):
        base, idx = (lhs, []) if lhs[0] == "var" else (lhs[1], lhs[2])
        if lhs[0] not in ("var", "idx") or base[0] != "var" or base[1] not in self.vars or self.vars[base[1]].kind != "local":
            raise StanSubsetError(f"line {line}: only model-block locals can be assigned")
        v = self.vars[base[1]]
        _, ic = self.flat_index(v, idx, line)
        cell = f"v_{v.name}" + (f"[{ic}]" if v.shape else "")
        dcell = f"d_{v.name}" + (f"[{ic}]" if v.shape else "")
        self_node = Node("local", name=v.name, idx=(ic if v.shape else None), deps=v.deps)
        if op in ("*=", "/="):
            rhs_node, op = _bin(op[0], self_node, rhs_node), "="
        self.emit("{")
        self.indent += 1
        val, leaves = self.emit_value_and_adjoints(rhs_node)
        if self.value_only:
            self.emit(f"{cell} {op} {val};")
        elif op == "=":
            reads_self = any(n.kind == "local" and n.name == v.name for n, _ in leaves)
            if reads_self and v.deps:        # the old sensitivities are inputs: build the new ones aside
                self.emit(f"double nd[{max(v.deps) + 1}];")
                self.emit_sensitivities(lambda k: f"nd[{k}]", leaves, v.deps, accumulate=False)
                for k in sorted(v.deps):
                    self.emit(f"{dcell}[{k}] = nd[{k}];")
            else:
                self.emit_sensitivities(lambda k: f"{dcell}[{k}]", leaves, v.deps, accumulate=False)
            self.emit(f"{cell} = {val};")
        else:
            sign = "" if op == "+=" else "-"
            if sign:
                leaves = [(n, f"(-({a}))") for n, a in leaves]
            self.emit_sensitivities(lambda k: f"{dcell}[{k}]", leaves, rhs_node.deps, accumulate=True)
            self.emit(f"{cell} {op} {val};")
        self.indent -= 1
        self.emit("}")

    def hoist_rng(self, e, pre, line, top=False):
        """`e` with every _rng call below it (innermost first; `top`: not `e` itself) replaced by a fresh local that a
        declaration appended to `pre` draws into: each call is evaluated once, as Stan does, however often the lowering
        reads the expression."""
        if isinstance(e, list):
            return [self.hoist_rng(x, pre, line) for x in e]
        if not (isinstance(e, tuple) and e and isinstance(e[0], str)) or not _has_rng(e):
            return e
        if e[0] != "call":
            return tuple(self.hoist_rng(x, pre, line) if isinstance(x, (tuple, list)) else x for x in e)
        new = ("call", e[1], [self.hoist_rng(a, pre, line) for a in e[2]], e[3])
        if top or not e[1].endswith("_rng"):
            return new
        dims, orient = self.shape(new)
        tmp = self.fresh_name("draw")
        self.vars[tmp] = _Var(tmp, "local", list(dims), "real", orient=orient)
        pre.append(("decl", (tmp, "real", [("num", float(d), True) for d in dims], None, None, new, line), line))
        return ("var", tmp, line)

    def hoist_rng_stmt(self, s):
        """Value-only mode: the statement with its _rng calls drawn ahead of it (a list), or None when it has nothing to
        draw first; cached by identity like lower_stmt."""
        key = id(s)
        if key not in self.rng_stmts:
            kind, line, out, pre = s[0], s[-1], None, []
            if kind in ("if", "while") and _has_rng(s[1]):
                raise StanSubsetError(f"line {line}: _rng calls inside a condition are outside the supported subset "
                                      f"(draw into a variable first)")
            if kind == "assign" and _has_rng(s):
                rhs = self.hoist_rng(s[3], pre, line, top=True)
                lhs = self.hoist_rng(s[1], pre, line)
                out = pre + [("assign", lhs, s[2], rhs, line)] if pre else None
            elif kind == "decl" and s[1][5] is not None and _has_rng(s[1][5]):
                d = s[1]
                init = self.hoist_rng(d[5], pre, line, top=True)
                out = pre + [("decl", (d[0], d[1], d[2], d[3], d[4], init, d[6]), line)] if pre else None
            self.rng_stmts[key] = (s, out)
        return self.rng_stmts[key][1]

    def scoped(self, stmts, emit):
        """statements() of a nested scope: a block, a loop body or a branch (value-only mode tracks its declarations)"""
        if not self.value_only:
            self.statements(stmts, emit)
            return
        self.scopes.append(set())
        try:
            self.statements(stmts, emit)
        finally:
            self.scopes.pop()

    def statements(self, stmts, emit=True):
        for s in stmts:
            kind, line = s[0], s[-1]
            if self.value_only:
                if kind in ("target", "tilde", "ptarget"):
                    raise StanSubsetError(f"line {line}: `target +=` and `~` are only allowed in the model block")
                drawn = self.hoist_rng_stmt(s)
                if drawn is not None:
                    self.statements(drawn, emit)
                    continue
            low = self.lower_stmt(s)
            if low is not None:
                self.statements(low, emit)
                continue
            if kind == "if":
                _, cond, then, other, _ = s
                if emit:
                    self.emit("{")
                    self.indent += 1
                    self.emit(f"if ({self.cond_text(cond, line)}) {{")
                    self.indent += 1
                self.scoped([then], emit)
                if other is not None:
                    if emit:
                        self.indent -= 1
                        self.emit("} else {")
                        self.indent += 1
                    self.scoped([other], emit)
                if emit:
                    self.indent -= 1
                    self.emit("}")
                    self.indent -= 1
                    self.emit("}")
                continue
            if kind == "print":      # output statements do not touch the density
                continue
            if kind == "reject":     # Stan throws; the reference maps the exception to logp = -inf (bridgestan.py:47-49)
                if emit:
                    self.emit("ok = false;")
                continue
            if kind == "while":      # the condition is re-evaluated at the top of every trip
                if emit:     # a loop that never ends would hang every lane of the device: after 2^24 trips the density is -inf
                    trip = self.new_tmp("trip")
                    self.emit(f"for (int {trip} = 0; ; ++{trip}) {{")
                    self.indent += 1
                    self.emit(f"if ({trip} >= (1 << 24)) {{ ok = false; break; }}")
                    self.emit(f"if (!{self.cond_text(s[1], line)}) break;")
                self.scoped([s[2]], emit)
                if emit:
                    self.indent -= 1
                    self.emit("}")
                continue
            if kind == "decl":
                name, base, shape, lo, hi, init, _ = s[1]
                if name in self.vars and self.vars[name].kind != "local":
                    raise StanSubsetError(f"line {line}: {name!r} shadows a data variable or parameter")
                if self.value_only:
                    if any(name in sc for sc in self.scopes):
                        raise StanSubsetError(f"line {line}: {name!r} is already declared")
                    self.scopes[-1].add(name)
                self.decl_lines.setdefault(name, line)
                dims = []
                for d in shape:
                    dv, _ = self.int_expr(d)
                    if dv is None:
                        raise StanSubsetError(f"line {line}: local array sizes must be constants")
                    dims.append(dv)
                if name not in self.vars:
                    self.vars[name] = _Var(name, "local", dims, base, orient=self.orients.get(name))
                if init is not None:     # one statement object per declaration: its lowering is cached by identity
                    first = self.decl_init.setdefault(id(s), ("assign", ("var", name, line), "=", init, line))
                    self.statements([first], emit)
            elif kind == "block":
                self.scoped(s[1], emit)
            elif kind == "for":
                _, var, lo, hi, body, _ = s
                (lov, loc), (hiv, hic) = self.int_expr(lo), self.int_expr(hi)
                cname = f"{var}_{len(self.loop_vars)}"
                if emit:
                    trip = (hiv - lov + 1) if (lov is not None and hiv is not None) else None
                    if var in self.rolled:          # literal bounds: never fully unrolled; others: nvcc's default
                        if trip is not None:
                            self.emit("#pragma unroll 1")
                    elif trip is not None and trip <= 16:
                        self.emit("#pragma unroll")
                    self.emit(f"for (int {cname} = {loc}; {cname} <= {hic}; ++{cname}) {{")
                    self.indent += 1
                self.loop_vars.append((var, cname))
                self.scoped(body, emit)
                self.loop_vars.pop()
                if emit:
                    self.indent -= 1
                    self.emit("}")
            elif kind == "target":
                if emit:
                    self.target_terms(s[1], line, drop_constant_terms=False)
            elif kind == "ptarget":      # one term of a `~` statement (vector densities): dropped when parameter-free
                if emit:
                    self.target_terms(s[1], line, drop_constant_terms=True)
            elif kind == "tilde":
                if emit:
                    _, lhs, dist, args, _ = s
                    if dist not in _DENSITIES:
                        raise StanSubsetError(f"line {line}: distribution {dist!r} is outside the supported subset")
                    self.target_terms(("call", dist + "_lpdf", [lhs] + args, line), line, drop_constant_terms=True)
            elif kind == "assign":
                _, lhs, op, rhs, _ = s
                node = self.real(rhs)
                if emit:
                    self.assign(lhs, op, node, line)
                else:      # activity analysis: the assigned local inherits the dependencies of its right-hand side
                    base = lhs if lhs[0] == "var" else lhs[1]
                    v = self.vars.get(base[1]) if base[0] == "var" else None
                    if v is None or v.kind != "local":
                        raise StanSubsetError(f"line {line}: only model-block locals can be assigned")
                    new = v.deps | node.deps
                    if new != v.deps:
                        v.deps = new
                        self.changed = True

    # ---- driver
    def run(self):
        # transformed data and transformed parameters (locals of the density; their declared bounds are validation only)
        # run ahead of the model
        program = self.declare_inputs()
        program += self.blocks.get("transformed parameters", [])
        program += self.blocks["model"]
        self.blocks["model"] = _demote_arrays(self.fuse_vector_densities(program)) if RESTRUCTURE else program
        # activity analysis (which coordinates can each local depend on): fixpoint over the statement list
        for _ in range(64):
            self.changed = False
            self.loop_vars = []
            self.statements(self.blocks["model"], emit=False)
            if not self.changed:
                break
        self.check_matrix_budget()
        # emission
        self.loop_vars = []
        body_start = len(self.lines)
        for v in self.vars.values():
            if v.kind == "local":
                dims = "".join(f"[{n}]" for n in ([v.size] if v.shape else []))
                self.emit(f"double v_{v.name}{dims}{' = {0.0}' if v.shape else ' = 0.0'};")
                if v.deps:
                    self.emit(f"double d_{v.name}{dims}[{max(v.deps) + 1}]{' = {{0.0}}' if v.shape else ' = {0.0}'};")
        self.statements(self.blocks["model"], emit=True)
        body = "\n".join(["        " + ln for ln in self.prologue] + self.lines[body_start:])
        return self.wrap(body)

    def run_gq(self, gq):
        """Value-only code of generated quantities (statements `gq`): transformed data and transformed parameters
        recomputed, then the block; its top-level declarations are the outputs.  -> (struct text, output names)"""
        program = self.declare_inputs() + self.blocks.get("transformed parameters", []) + list(gq)
        outputs = [st[1] for st in gq if st[0] == "decl"]
        for name, base, shape, lo, hi, init, line in outputs:
            if self.orients.get(name) == "mat":
                raise StanSubsetError(f"line {line}: matrix outputs of generated quantities are outside the supported "
                                      f"subset")
        self.loop_vars = []
        self.statements(program, emit=True)
        self.check_matrix_budget()
        body = self.lines
        self.lines = []
        for v in self.vars.values():         # locals start as NaN, as in Stan
            if v.kind == "local":
                self.emit(f"double v_{v.name}{f'[{v.size}]' if v.shape else ''};")
                self.emit(f"for (int i = 0; i < {v.size}; ++i) v_{v.name}{'[i]' if v.shape else ''} = NAN;"
                          if v.shape else f"v_{v.name} = NAN;")
        names, copy = [], []
        for name, *_ in outputs:
            v = self.vars[name]
            copy.append(f"for (int j = 0; j < {v.size}; ++j) out[{len(names)} + j] = v_{name}[j];" if v.shape else
                        f"out[{len(names)}] = v_{name};")
            names += [name if not v.shape else f"{name}.{'.'.join(str(i + 1) for i in _unravel(j, v.shape))}"
                      for j in range(v.size)]
        if len(names) > self.MAX_GQ:
            raise StanSubsetError(f"{len(names)} generated quantities; the generated kernels support up to {self.MAX_GQ}")
        return self.wrap_gq("\n".join(["        " + ln for ln in self.prologue] + self.lines + body), copy, len(names)), names

    def check_matrix_budget(self):
        """Refuses a program whose matrix locals, values and tangents, take more than MAX_MATRIX_BYTES a thread (named
        with the declaration that crosses the budget)."""
        total = 0
        for v in self.vars.values():
            if v.kind == "local" and v.orient == "mat":
                nd = max(v.deps) + 1 if v.deps else 0
                total += 8 * v.size * (1 + nd)
                if total > self.MAX_MATRIX_BYTES:
                    raise StanSubsetError(
                        f"line {self.decl_lines.get(v.name, '?')}: matrix locals take {total} bytes a thread up to "
                        f"{v.name.split('__')[0]!r} ({' x '.join(map(str, v.shape))}, {1 + nd} double(s) an entry with "
                        f"its tangents); the generated kernels allow up to {self.MAX_MATRIX_BYTES}")

    def fold_data_cholesky(self, st):
        """`matrix[K, K] L = cholesky_decompose(S);` in transformed data, with S a data matrix and L assigned nowhere
        else: L becomes data, factored now (True), instead of a local factored in every evaluation"""
        if st[0] != "decl" or self.value_only:
            return False
        name, _, shape, _, _, init, line = st[1]
        if not (init is not None and init[0] == "call" and init[1] == "cholesky_decompose" and len(init[2]) == 1
                and init[2][0][0] == "var" and self.orients.get(name) == "mat"):
            return False
        src = self.vars.get(init[2][0][1])
        if src is None or src.kind != "data" or src.orient != "mat":
            return False
        others = [s for blk in ("transformed data", "transformed parameters", "model") for s in self.blocks.get(blk, [])
                  if s is not st]
        if name in _assigned_names(others, set()):
            return False
        n = self.square_dim(init[2][0], "cholesky_decompose", line)
        if [self.int_expr(d)[0] for d in shape] != [n, n]:
            raise StanSubsetError(f"line {line}: assignment of a {n} x {n} factor to {name!r} of size "
                                  f"{[self.int_expr(d)[0] for d in shape]}")
        self.data_matrix(name, n, self.cholesky_of_data(src.name, line))
        return True

    def declare_inputs(self):
        """Data, parameters and the integer constants of transformed data -> the other transformed data statements."""
        # data block
        for name, base, shape, lo, hi, init, line in self.blocks["data"]:
            dims = [self.int_expr(d)[0] for d in shape]
            if name == "phi" and name not in self.data_in:
                self.data_in[name] = 1.0
            if name not in self.data_in:
                raise StanSubsetError(f"line {line}: data variable {name!r} is missing from the data")
            val = self.data_in[name]
            if dims:
                flat = [float(z) for z in _flatten(val)]
                n = 1
                for d in dims:
                    n *= d
                if len(flat) != n:
                    raise StanSubsetError(f"data {name!r}: expected {n} values, found {len(flat)}")
                if name in self.ctypes:
                    self.check_vector_data(name, self.ctypes[name], flat, dims[-1], line)
                v = _Var(name, "data", dims, base, offset=len(self.blob), value=flat, orient=self.orients.get(name))
                self.blob += flat
            else:
                v = _Var(name, "data", [], base, value=(int(val) if base == "int" else float(val)))
            self.vars[name] = v
        # parameters block
        # parameters block: the density sees constrained values c[0 .. CDIM) (param leaves index them); a scalar
        # coordinate has one of each, a simplex[K] K - 1 unconstrained coordinates and K constrained values
        off, uoff = 0, 0
        for name, base, shape, lo, hi, init, line in self.blocks["parameters"]:
            if base != "real":
                raise StanSubsetError(f"line {line}: parameters must be real")
            dims = [self.int_expr(d)[0] for d in shape]
            lov = None if lo is None else self._const_value(lo, line)
            hiv = None if hi is None else self._const_value(hi, line)
            if self.orients.get(name) == "mat":
                raise StanSubsetError(f"line {line}: matrix parameters are outside the supported subset (BridgeStan orders them "
                                      f"column-major; declare an array of vectors)")
            v = _Var(name, "param", dims, "real", offset=off, lower=lov, upper=hiv, orient=self.orients.get(name))
            self.vars[name] = v
            for j in range(v.size):
                self.param_names.append(name if not dims else f"{name}.{'.'.join(str(i + 1) for i in _unravel(j, dims))}")
            kind = self.ctypes.get(name)
            if kind is None:
                kind = "none" if (lov is None and hiv is None) else "both" if (lov is not None and hiv is not None) else \
                    "lower" if lov is not None else "upper"
                for j in range(v.size):
                    self.transforms.append((kind, lov, hiv))
                    self.blocks_of.append((kind, lov, hiv, uoff + j, off + j, 1))
                self.param_unc_names += self.param_names[len(self.param_names) - v.size:]
                uoff += v.size
            else:
                K = dims[-1]
                if K < (2 if kind == "simplex" else 1):
                    raise StanSubsetError(f"line {line}: a {kind} needs at least {2 if kind == 'simplex' else 1} element(s)")
                nu = K - 1 if kind == "simplex" else K
                outer = dims[:-1]
                for j in range(v.size // K):
                    self.blocks_of.append((kind, None, None, uoff, off + j * K, K))
                    for i in range(nu):
                        self.transforms.append((kind, None, None))
                        self.param_unc_names.append(f"{name}.{'.'.join(str(q + 1) for q in _unravel(j, outer) + [i])}"
                                                    if outer else f"{name}.{i + 1}")
                    uoff += nu
            off += v.size
        self.dim, self.cdim = uoff, off
        if not (1 <= self.dim <= self.MAX_DIM):
            raise StanSubsetError(f"{self.dim} unconstrained parameters; the generated kernels support 1..{self.MAX_DIM}")
        if self.cdim > 2 * self.MAX_DIM:
            raise StanSubsetError(f"{self.cdim} constrained parameter values; the generated kernels support up to "
                                  f"{2 * self.MAX_DIM}")
        # transformed data: integer scalars folded now, everything else computed like a parameter-free local
        program = []
        for st in self.blocks.get("transformed data", []):
            if st[0] == "decl" and st[1][1] == "int":
                name, _, shape, _, _, init, line = st[1]
                if shape or init is None:
                    raise StanSubsetError(f"line {line}: transformed data integers must be scalars defined where they are declared")
                self.vars[name] = _Var(name, "data", [], "int", value=self.int_expr(init)[0])
                if self.vars[name].value is None:
                    raise StanSubsetError(f"line {line}: {name!r} is not a constant")
            elif not self.fold_data_cholesky(st):
                program.append(st)
        return program

    @staticmethod
    def check_vector_data(name, kind, flat, K, line):
        """Stan validates constrained data when it reads it: rows of a simplex are >= 0 and sum to 1 (within 1e-8),
        ordered rows increase strictly, positive_ordered rows also start above 0."""
        for r in range(len(flat) // K):
            row = flat[r * K:(r + 1) * K]
            if kind == "simplex":
                bad = any(not (z >= 0.0) for z in row) or not abs(math.fsum(row) - 1.0) <= 1e-8
            else:
                bad = any(not (b > a) for a, b in zip(row, row[1:])) or (kind == "positive_ordered" and not row[0] > 0.0)
            if bad:
                raise StanSubsetError(f"line {line}: data {name!r} is not a valid {kind} (row {r + 1}: {row})")

    def _const_value(self, e, line):
        n = self.real(e)
        if n.kind != "const":
            raise StanSubsetError(f"line {line}: parameter bounds must be constants")
        return n.val

    _VECTOR_CALL = {"simplex": "simplex_{0}<{1}>", "ordered": "ordered_{0}<{1}, false>",
                    "positive_ordered": "ordered_{0}<{1}, true>"}

    def wrap(self, body):
        D, C = self.dim, self.cdim
        pro, con, pull = [], [], []
        for kind, lo, hi, u, k, K in self.blocks_of:
            if kind == "none":
                pro.append(f"c[{k}] = x[{u}]; dc[{k}] = 1.0;")
                con.append(f"out[{k}] = x[{u}];")
                pull.append(f"g[{u}] = gc[{k}];")
            elif kind == "lower":
                pro.append(f"{{ const double e = exp(x[{u}]); c[{k}] = {self.lit(lo)} + e; dc[{k}] = e; A += x[{u}]; gA[{k}] += 1.0; "
                           f"ok = ok && e > 0.0 && e < INFINITY; }}")
                con.append(f"out[{k}] = {self.lit(lo)} + exp(x[{u}]);")
                pull.append(f"g[{u}] = gc[{k}];")
            elif kind == "upper":
                pro.append(f"{{ const double e = exp(x[{u}]); c[{k}] = {self.lit(hi)} - e; dc[{k}] = -e; A += x[{u}]; gA[{k}] += 1.0; "
                           f"ok = ok && e > 0.0 && e < INFINITY; }}")
                con.append(f"out[{k}] = {self.lit(hi)} - exp(x[{u}]);")
                pull.append(f"g[{u}] = gc[{k}];")
            elif kind == "both":
                w = self.lit(hi - lo)
                pro.append(f"{{ const double s = smcgen_inv_logit(x[{u}]); c[{k}] = {self.lit(lo)} + {w} * s; dc[{k}] = {w} * s * (1.0 - s); "
                           f"A += log({w}) + log(s) + log1p(-s); gA[{k}] += 1.0 - 2.0 * s; ok = ok && s > 0.0 && s < 1.0; }}")
                con.append(f"out[{k}] = {self.lit(lo)} + {w} * smcgen_inv_logit(x[{u}]);")
                pull.append(f"g[{u}] = gc[{k}];")
            else:        # a vector type: the body sees its K values as K independent leaves (dc = 1), pulled back below
                fn = "smcb::stan::" + self._VECTOR_CALL[kind]
                pro.append(f"A += {fn.format('constrain', K)}(&x[{u}], &c[{k}], ok);")
                pro.append(f"for (int j = 0; j < {K}; ++j) dc[{k} + j] = 1.0;")
                con.append(f"{fn.format('constrain', K)}(&x[{u}], &out[{k}], ok);")
                pull.append(f"{fn.format('pullback', K)}(&x[{u}], " + (f"&c[{k}], " if kind == "simplex" else "")
                            + f"&gc[{k}], &g[{u}]);")
        if C == D and all(b[0] in ("none", "lower", "upper", "both") for b in self.blocks_of):
            tail = f"""#pragma unroll
        for (int k = 0; k < {D}; ++k) g[k] = gA[k] + phi * gB[k];"""
        else:            # gradient over the constrained values, then one pullback per transform (log-Jacobian included)
            tail = f"""double gc[{C}];
#pragma unroll
        for (int k = 0; k < {C}; ++k) gc[k] = gA[k] + phi * gB[k];
        """ + "\n        ".join(pull)
        staged = len(self.blob) if len(self.blob) <= 4096 else 0
        text = f"""// GENERATED by smcnuts/model/stan_codegen.py -- do not edit.  Model struct with the interface of csrc/models.cuh.
#pragma once
#include <cmath>
#include "stan_transforms.cuh"
#ifndef SMCGEN_HELPERS
#define SMCGEN_HELPERS
SMCB_HD double smcgen_inv_logit(double z) {{ return z >= 0.0 ? 1.0 / (1.0 + exp(-z)) : exp(z) / (1.0 + exp(z)); }}
SMCB_HD double smcgen_log1p_exp(double z) {{ return (z > 0.0 ? z : 0.0) + log1p(exp(-fabs(z))); }}
// d/dx lgamma(x) for x > 0: upward recurrence to x >= 10, then the asymptotic series (next term 691/32760 x^-12 < 3e-14)
SMCB_HD double smcgen_digamma(double x) {{
    if (!(x > 0.0)) return NAN;          // Stan rejects such shapes; also keeps the recurrence below bounded (10 trips at most)
    double r = 0.0;
    while (x < 10.0) {{ r -= 1.0 / x; x += 1.0; }}
    const double f = 1.0 / (x * x);
    return r + log(x) - 0.5 / x
           - f * (1.0 / 12 - f * (1.0 / 120 - f * (1.0 / 252 - f * (1.0 / 240 - f * (1.0 / 132)))));
}}
#endif
struct {self.struct_name} {{
    static constexpr int DMAX = {D}, STATIC_D = {D}, CDIM = {C};
    static constexpr int GROUP = 1, NLOC = {D}, STATIC_NL = {D};
    static constexpr bool STAGE = false;
    static constexpr int NDATA = {len(self.blob)}, NSTAGED = {staged};
    const double* data;
    SMCB_HD explicit {self.struct_name}(const smcb::ModelDesc& d, const double* staged) : data(NSTAGED ? staged : d.data) {{}}
    SMCB_HD static constexpr int dim_of(const smcb::ModelDesc&) {{ return {D}; }}
    SMCB_HD constexpr int dim() const {{ return {D}; }}
    SMCB_HD constexpr int nloc() const {{ return {D}; }}
    static int staged_doubles(const smcb::ModelDesc&) {{ return NSTAGED; }}

    // A = log prior + log Jacobian (everything not multiplied by phi), B = the phi-scaled part, g = grad A + phi * grad B
    SMCB_HD void eval(const double (&x)[DMAX], double phi, double& A_out, double& B_out, double (&g)[DMAX]) const {{
        double A = 0.0, B = 0.0, gA[{C}] = {{0.0}}, gB[{C}] = {{0.0}}, c[{C}], dc[{C}];
        bool ok = true;
        {(chr(10) + '        ').join(pro)}
{body}
        if (!ok) A = -INFINITY;      // a constrained value under- or overflowed: Stan throws, the reference maps it to -inf
        A_out = A; B_out = B;
        {tail}
    }}

    // Stan's constraining transforms of the declared parameters, in declaration order: out[0 .. CDIM)
    SMCB_HD static void constrain(const double (&x)[DMAX], double* out) {{
        bool ok = true;
        {(chr(10) + '        ').join(con)}
        (void)ok;
    }}
}};
"""
        return text

    def wrap_gq(self, body, copy, G):
        """The generated-quantities struct (`<model struct>GQ`, text included after the model struct): `copy` moves
        the outputs to out[0 .. GDIM)."""
        S = self.struct_name
        return f"""// GENERATED by smcnuts/model/stan_codegen.py -- do not edit.  Generated quantities of {S} (included after it).
#pragma once
#include "stan_rng.cuh"
struct {S}GQ {{
    static constexpr int DMAX = {self.dim}, CDIM = {self.cdim}, GDIM = {G};
    const double* data;
    SMCB_HD explicit {S}GQ(const smcb::ModelDesc& d) : data(d.data) {{}}

    // out[0 .. GDIM) of the unconstrained row x, drawing from rng; all NaN when a draw's arguments are invalid (Stan
    // throws) or the block rejects
    SMCB_HD void generated_quantities(const double (&x)[DMAX], smcb::stan::Rng& rng, double* out) const {{
        double c[CDIM];
        {S}::constrain(x, c);
        bool ok = true;
{body}
        if (ok && rng.ok) {{
            {(chr(10) + '            ').join(copy)}
        }} else {{
            for (int k = 0; k < GDIM; ++k) out[k] = NAN;
        }}
    }}
}};
"""


def _flatten(v):
    if isinstance(v, (list, tuple)):
        for z in v:
            yield from _flatten(z)
    elif hasattr(v, "tolist") and not isinstance(v, (int, float)):
        yield from _flatten(v.tolist())
    else:
        yield v


def _unravel(j, dims):
    out = []
    for n in reversed(dims):
        out.append(j % n)
        j //= n
    return list(reversed(out))


def load_data(data_path):
    """Read a Stan data JSON (the shipped PRMwCD.json is truncated after `"phi": `: repaired as the reference's _update_phi
    would rewrite it, with phi = 1)."""
    if data_path is None or str(data_path) == "None":
        return {}
    raw = Path(data_path).read_text()
    try:
        return json.loads(raw)
    except json.JSONDecodeError:
        return json.loads(raw + " 1.0}")


def generate(stan_text, data, struct_name="GenModel"):
    """Stan program text + data dict -> GeneratedSource."""
    import hashlib
    parser = _Parser(stan_text)
    blocks = parser.program()
    gq_blocks = dict(blocks)             # run() rewrites the model block in place
    g = _Gen(blocks, data, struct_name, parser.orients, parser.ctypes)
    text = g.run()
    gq_names, gq_error = [], blocks.get("generated quantities error")
    gq_text = g.wrap_gq("", [], 0)
    if gq_error is None and blocks.get("generated quantities"):
        try:
            q = _Gen(gq_blocks, data, struct_name, dict(parser.gq_orients), dict(parser.gq_ctypes), value_only=True)
            gq_text, gq_names = q.run_gq(blocks["generated quantities"])
        except StanSubsetError as e:
            gq_error = str(e)
    digest = hashlib.sha256((text + gq_text + repr(g.blob)).encode()).hexdigest()[:16]
    return GeneratedSource(struct_name, text, g.dim, g.blob, g.param_names, g.transforms, digest, g.cdim, g.param_unc_names,
                           gq_text, gq_names, gq_error)
