"""ctypes mirror of include/rafting_b200.h plus numpy-backed batch builders.

The structs here must stay field-for-field identical to the header; tests/test_abi.py checks the
sizes against values compiled into the shared library.  The batch classes (Inbox / Outbox) own the
column memory as numpy arrays (host memory) and hand out the C structs that point into them.

Reference surfaces the columns stand for are documented in the header; in short an Inbox row is
one turn of every group's ContextEventLoop (M/support/EventLoop.java:41-101): at most one group op
(an inbound RPC, a timer expiry or a client submit) followed by one Async callback per follower lane.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

ABI_VERSION = 2
INBOX_NO_REQUESTS = 1
INBOX_COMPACT_GROUPS = 2
CFG_STRICT_CANDIDATE_VOTE = 1
CFG_LENIENT_FOLLOWER_COMMIT = 2
TERM_RUNS = 8
MAX_REPLICAS = 33
I64_MAX = (1 << 63) - 1

ROLE_FOLLOWER, ROLE_CANDIDATE, ROLE_LEADER = 0, 1, 2
ROLE_NAMES = {0: "Follower", 1: "Candidate", 2: "Leader"}

OP_NONE, OP_SUBMIT, OP_TIMEOUT, OP_AE_REQUEST, OP_PREVOTE_REQ, OP_VOTE_REQ, OP_IS_REQUEST, OP_FLUSH = range(8)
EV_NONE, EV_AE_ACK, EV_IS_ACK, EV_PV_REPLY, EV_RV_REPLY = range(5)
OUT_OK, OUT_ERROR, OUT_CANCELED = 0, 1, 2
PLAN_NONE, PLAN_AE, PLAN_IS, PLAN_SKIP_INFLIGHT, PLAN_UNAVAILABLE = range(5)
BALLOT_NONE, BALLOT_PREVOTE, BALLOT_VOTE = range(3)

ERR_NAMES = {
    0: "OK", 1: "MATCH_ROLLBACK", 2: "IMPOSSIBLE_REPL", 3: "COMMIT_ROLLBACK", 4: "TRY_COMMIT_FAILED",
    5: "LEADER_SELF_AE", 6: "TWO_LEADERS", 7: "LEADER_VOTE_SELF", 8: "FOLLOWER_TWO_LEADERS",
    9: "INDEX_TERM_ZERO", 10: "EPOCH_TERM_MISMATCH", 11: "IMPOSSIBLE_LOG", 12: "CANDIDATE_SELF_RV",
    13: "CANDIDATE_VOTE_SELF", 14: "IS_BEFORE_AE", 15: "LEADER_UNCHANGED", 16: "BALLOT_MISMATCH",
    17: "LOG_NOT_FOLLOW_EPOCH", 18: "LOG_NOT_CONTINUOUS", 19: "LOG_START", 20: "LOG_VACANCY",
    21: "FLUSH_RANGE", 22: "TERM_RUNS_OVERFLOW", 23: "LOG_SHAPE", 24: "NOT_LEADER", 25: "NOT_READY",
    26: "BAD_EVENT", 27: "CLOSED_GROUP",
}
ERR = {v: k for k, v in ERR_NAMES.items()}

I64X2 = np.dtype([("x", "<i8"), ("y", "<i8")])


class Cfg(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("replicas", C.c_uint32), ("local_slot", C.c_uint32),
        ("max_groups", C.c_uint32), ("max_rows", C.c_uint32), ("entry_pool_cap", C.c_uint32),
        ("pre_vote", C.c_int32), ("avail_critical_point", C.c_int32),
        ("recovery_cool_down_ms", C.c_int64), ("heartbeat_ms", C.c_int64), ("broadcast_ms", C.c_int64),
        ("election_ms", C.c_int64), ("timer_seed", C.c_uint64),
        ("device", C.c_int32), ("flags", C.c_uint32),
    ]


def make_cfg(replicas=3, local_slot=0, max_groups=1024, max_rows=16, entry_pool_cap=0, pre_vote=True,
             avail_critical_point=0, recovery_cool_down_ms=0, heartbeat_ms=300, broadcast_ms=150,
             election_ms=900, timer_seed=0x5EED, device=0, flags=0) -> Cfg:
    """Defaults follow the reference's test config R/raft1.xml:8-14 (tick 300 ms, heartbeat 1,
    election 3, broadcast 0.5, pre-vote true)."""
    c = Cfg()
    c.struct_size = C.sizeof(Cfg)
    c.replicas, c.local_slot, c.max_groups, c.max_rows = replicas, local_slot, max_groups, max_rows
    c.entry_pool_cap = entry_pool_cap
    c.pre_vote = 1 if pre_vote else 0
    c.avail_critical_point = avail_critical_point
    c.recovery_cool_down_ms = recovery_cool_down_ms
    c.heartbeat_ms, c.broadcast_ms, c.election_ms = heartbeat_ms, broadcast_ms, election_ms
    c.timer_seed = timer_seed
    c.device = device
    c.flags = flags
    return c


class InboxC(C.Structure):
    _fields_ = [
        ("rows", C.c_uint32), ("n_active", C.c_uint32),
        ("gids", C.c_void_p), ("row_now", C.c_void_p),
        ("op_meta", C.c_void_p), ("op_nr", C.c_void_p), ("op_ab", C.c_void_p), ("op_cd", C.c_void_p),
        ("op_e", C.c_void_p), ("ent_terms", C.c_void_p),
        ("ent_count", C.c_uint32), ("flags", C.c_uint32),
        ("ev_meta", C.c_void_p), ("ev_tn", C.c_void_p), ("ev_el", C.c_void_p),
    ]


class OutboxC(C.Structure):
    _fields_ = [
        ("rep_meta", C.c_void_p), ("rep_term", C.c_void_p),
        ("plan_meta", C.c_void_p), ("plan_pp", C.c_void_p), ("plan_lc", C.c_void_p), ("plan_epoch", C.c_void_p),
        ("ballot_meta", C.c_void_p), ("ballot_term", C.c_void_p), ("ballot_last", C.c_void_p),
        ("commit_index", C.c_void_p), ("current_term", C.c_void_p), ("role_word", C.c_void_p),
        ("incarnation", C.c_void_p), ("err_word", C.c_void_p), ("last_entry", C.c_void_p),
    ]


class LeaseC(C.Structure):
    _fields_ = [("inbox", InboxC), ("outbox", OutboxC), ("generation", C.c_uint32), ("_pad", C.c_uint32)]


class GroupInit(C.Structure):
    _fields_ = [
        ("term", C.c_int64), ("ballot", C.c_int32), ("_pad", C.c_int32),
        ("epoch_index", C.c_int64), ("epoch_term", C.c_int64),
        ("first_index", C.c_int64), ("last_index", C.c_int64), ("last_term", C.c_int64),
        ("commit_index", C.c_int64), ("now_ms", C.c_int64), ("rand_ms", C.c_int64),
    ]


GROUP_INIT_DTYPE = np.dtype([
    ("term", "<i8"), ("ballot", "<i4"), ("_pad", "<i4"), ("epoch_index", "<i8"), ("epoch_term", "<i8"),
    ("first_index", "<i8"), ("last_index", "<i8"), ("last_term", "<i8"), ("commit_index", "<i8"),
    ("now_ms", "<i8"), ("rand_ms", "<i8"),
])
assert GROUP_INIT_DTYPE.itemsize == C.sizeof(GroupInit)


class FollowerState(C.Structure):
    _fields_ = [
        ("last_request", C.c_int64), ("request_success", C.c_int64), ("request_failure", C.c_int64),
        ("request_in_flight", C.c_int32), ("recent_rejection", C.c_int32), ("recent_failure", C.c_int32),
        ("pending_installation", C.c_int32),
        ("last_epoch", C.c_int64), ("next_index", C.c_int64), ("match_index", C.c_int64),
    ]


class GroupState(C.Structure):
    _fields_ = [
        ("alive", C.c_uint32), ("role", C.c_uint32), ("current_term", C.c_int64),
        ("voted_for", C.c_int32), ("current_leader", C.c_int32),
        ("incarnation", C.c_uint32), ("timeout_detected", C.c_uint32),
        ("leader_prepared", C.c_uint32), ("votes", C.c_int32),
        ("elected_inc", C.c_uint32), ("elected_aborted", C.c_uint32), ("elected_term", C.c_int64),
        ("timer", C.c_int64), ("commit_index", C.c_int64),
        ("epoch_index", C.c_int64), ("epoch_term", C.c_int64),
        ("first_index", C.c_int64), ("last_index", C.c_int64), ("last_term", C.c_int64),
        ("term_runs", C.c_uint32), ("err_word", C.c_uint32), ("log_digest", C.c_uint64),
        ("n_followers", C.c_uint32), ("_pad", C.c_uint32),
        ("followers", FollowerState * (MAX_REPLICAS - 1)),
    ]

    def as_dict(self) -> dict:
        d = {}
        for name, _ in self._fields_:
            if name in ("_pad", "followers"):
                continue
            d[name] = getattr(self, name)
        d["followers"] = [
            {n: getattr(self.followers[f], n) for n, _ in FollowerState._fields_}
            for f in range(self.n_followers)
        ]
        return d

    def raw(self) -> bytes:
        return bytes(self)


def op_make(kind: int, peer: int = 0, count: int = 0) -> int:
    return (kind & 0xFF) | ((peer & 0xFF) << 8) | ((count & 0xFFFF) << 16)


def evm_make(kind: int, outcome: int = OUT_OK, success: bool = True, incarnation: int = 0) -> int:
    return (kind & 0xF) | ((outcome & 3) << 4) | ((1 if success else 0) << 6) | ((incarnation & 0xFFFFFFFF) << 32)


def _ptr(a):
    return None if a is None else a.ctypes.data


class Inbox:
    """Host-memory inbox for one step: `rows` rows over `n` groups with F follower lanes."""

    def __init__(self, rows: int, n: int, F: int, ent_cap: int = 0, gids=None, with_ops=True, with_events=True,
                 sweep=False):
        self.rows, self.n, self.F = rows, n, F
        self.gids = None if gids is None else np.ascontiguousarray(gids, dtype=np.uint32)
        self.row_now = np.zeros(rows, dtype=np.int64) if sweep else None
        if with_ops:
            self.op_meta = np.zeros((rows, n), dtype=np.uint64)
            self.op_nr = np.zeros((rows, n), dtype=I64X2)
            self.op_ab = np.zeros((rows, n), dtype=I64X2)
            self.op_cd = np.zeros((rows, n), dtype=I64X2)
            self.op_e = np.zeros((rows, n), dtype=np.int64)
        else:
            self.op_meta = self.op_nr = self.op_ab = self.op_cd = self.op_e = None
        self.ent_terms = np.zeros(max(ent_cap, 1), dtype=np.int64)
        self.ent_count = 0
        self.flags = 0
        if with_events:
            self.ev_meta = np.zeros((rows, n, F), dtype=np.uint64)
            self.ev_tn = np.zeros((rows, n, F), dtype=I64X2)
            self.ev_el = np.zeros((rows, n, F), dtype=I64X2)
        else:
            self.ev_meta = self.ev_tn = self.ev_el = None

    # ---- group ops -------------------------------------------------------------------------
    def _op(self, r, i, kind, now, rand=0, peer=0, count=0, a=0, b=0, c=0, d=0, e=0, ent=0):
        self.op_meta[r, i] = op_make(kind, peer, count) | (ent << 32)
        self.op_nr[r, i] = (now, rand)
        self.op_ab[r, i] = (a, b)
        self.op_cd[r, i] = (c, d)
        self.op_e[r, i] = e

    def submit(self, r, i, now, count=1, unavail=0):
        self._op(r, i, OP_SUBMIT, now, count=count, a=unavail)

    def timeout(self, r, i, now, rand=0, unavail=0):
        self._op(r, i, OP_TIMEOUT, now, rand=rand, a=unavail)

    def ae_request(self, r, i, now, leader, term, prev_index, prev_term, entry_terms=(), leader_commit=0,
                   first_index=None, rand=0):
        n = len(entry_terms)
        off = self.ent_count
        if n:
            if off + n > len(self.ent_terms):
                self.ent_terms = np.concatenate([self.ent_terms, np.zeros(max(n, len(self.ent_terms)), np.int64)])
            self.ent_terms[off:off + n] = entry_terms
            self.ent_count += n
        first = prev_index + 1 if first_index is None else first_index
        self._op(r, i, OP_AE_REQUEST, now, rand=rand, peer=leader, count=n, a=term, b=prev_index, c=prev_term,
                 d=leader_commit, e=first, ent=off)

    def prevote_request(self, r, i, now, candidate, term, last_index, last_term, rand=0):
        self._op(r, i, OP_PREVOTE_REQ, now, rand=rand, peer=candidate, a=term, b=last_index, c=last_term)

    def vote_request(self, r, i, now, candidate, term, last_index, last_term, rand=0):
        self._op(r, i, OP_VOTE_REQ, now, rand=rand, peer=candidate, a=term, b=last_index, c=last_term)

    def is_request(self, r, i, now, leader, term, last_included_index, last_included_term, host_result, rand=0):
        self._op(r, i, OP_IS_REQUEST, now, rand=rand, peer=leader, a=term, b=last_included_index,
                 c=last_included_term, d=1 if host_result else 0)

    def flush(self, r, i, now, index, term):
        self._op(r, i, OP_FLUSH, now, b=index, c=term)

    # ---- lane events -----------------------------------------------------------------------
    def ack(self, r, i, f, now, incarnation, resp_term, success, epoch_at_send, last_at_send, outcome=OUT_OK,
            snapshot=False):
        self.ev_meta[r, i, f] = evm_make(EV_IS_ACK if snapshot else EV_AE_ACK, outcome, success, incarnation)
        self.ev_tn[r, i, f] = (resp_term, now)
        self.ev_el[r, i, f] = (epoch_at_send, last_at_send)

    def vote_reply(self, r, i, f, now, incarnation, resp_term, granted, outcome=OUT_OK, pre=False):
        self.ev_meta[r, i, f] = evm_make(EV_PV_REPLY if pre else EV_RV_REPLY, outcome, granted, incarnation)
        self.ev_tn[r, i, f] = (resp_term, now)

    def as_c(self) -> InboxC:
        c = InboxC()
        c.rows = self.rows
        c.n_active = 0 if self.gids is None else len(self.gids)
        c.gids = _ptr(self.gids)
        c.row_now = _ptr(self.row_now)
        c.op_meta, c.op_nr, c.op_ab, c.op_cd, c.op_e = map(_ptr, (self.op_meta, self.op_nr, self.op_ab, self.op_cd, self.op_e))
        c.ent_terms = _ptr(self.ent_terms)
        c.ent_count = self.ent_count
        c.flags = self.flags
        c.ev_meta, c.ev_tn, c.ev_el = map(_ptr, (self.ev_meta, self.ev_tn, self.ev_el))
        return c


class Outbox:
    """Host-memory outbox.  Row columns are [rows, n(, F)]; group columns are [G] indexed by gid."""

    ROW_COLS = (("rep_meta", np.uint32, False), ("rep_term", np.int64, False),
                ("plan_meta", np.uint64, True), ("plan_pp", I64X2, True), ("plan_lc", I64X2, True),
                ("plan_epoch", np.int64, True),
                ("ballot_meta", np.uint64, False), ("ballot_term", np.int64, False), ("ballot_last", I64X2, False))
    GROUP_COLS = (("commit_index", np.int64), ("current_term", np.int64), ("role_word", np.uint32),
                  ("incarnation", np.uint32), ("err_word", np.uint32), ("last_entry", I64X2))

    def __init__(self, rows: int, n: int, F: int, G: int):
        self.rows, self.n, self.F, self.G = rows, n, F, G
        for name, dt, lane in self.ROW_COLS:
            shape = (rows, n, F) if lane else (rows, n)
            setattr(self, name, np.zeros(shape, dtype=dt))
        for name, dt in self.GROUP_COLS:
            setattr(self, name, np.zeros(G, dtype=dt))

    def as_c(self) -> OutboxC:
        c = OutboxC()
        for name, _, _ in self.ROW_COLS:
            setattr(c, name, _ptr(getattr(self, name)))
        for name, _ in self.GROUP_COLS:
            setattr(c, name, _ptr(getattr(self, name)))
        return c

    def row_bytes(self) -> bytes:
        return b"".join(getattr(self, name).tobytes() for name, _, _ in self.ROW_COLS)

    def payload_masks(self) -> dict:
        """Where each payload row column holds a value, as its meta column says: rep_term where a reply exists, plan_*
        where a plan exists, ballot_* where a ballot exists.  Meta columns are always valid and have no entry."""
        pm = (self.plan_meta & np.uint64(0xF)) != 0
        bm = self.ballot_meta != 0
        return {"rep_term": (self.rep_meta & 1) != 0, "plan_pp": pm, "plan_lc": pm, "plan_epoch": pm,
                "ballot_term": bm, "ballot_last": bm}

    def equal(self, other: "Outbox", gids=None) -> list[str]:
        """Names of columns that differ.  Payload columns are compared only where payload_masks() says they
        are valid; group columns only on `gids` if given."""
        bad = []

        def cmp(name, mask=None):
            a, b = getattr(self, name), getattr(other, name)
            if mask is not None:
                a, b = a[mask], b[mask]
            if not np.array_equal(a, b):
                bad.append(name)

        masks = self.payload_masks()
        for name, _, _ in self.ROW_COLS:
            cmp(name, masks.get(name))
        for name, _ in self.GROUP_COLS:
            cmp(name, gids)
        return bad


def role_of(role_word: int) -> int:
    return role_word & 3


def voted_for_of(role_word: int) -> int:
    return ((role_word >> 8) & 0xFF) - 1


def leader_of(role_word: int) -> int:
    return ((role_word >> 16) & 0xFF) - 1


# ---- compact host path (include/rafting_b200.h "COMPACT host path") --------------------------------------------------
CEV_ESCAPED, CTAG_NONE = 15, 63
CESC_PLAN, CESC_BALLOT, CESC_REPLY = 1, 2, 3
CESC_IN = np.dtype([("slot", "<u4"), ("_pad", "<u4"), ("ev_meta", "<u8"), ("term", "<i8"), ("now_ms", "<i8"),
                    ("epoch_at_send", "<i8"), ("last_at_send", "<i8")])
CESC_OUT = np.dtype([("kind", "<u4"), ("slot", "<u4"), ("meta", "<u8"), ("a", "<i8"), ("b", "<i8"), ("c", "<i8"), ("d", "<i8"), ("e", "<i8")])
assert CESC_IN.itemsize == 48 and CESC_OUT.itemsize == 56


class CInboxC(C.Structure):
    _fields_ = [("rows", C.c_uint32), ("n_esc", C.c_uint32),
                ("row_base", C.c_void_p), ("op_c", C.c_void_p), ("op_unavail", C.c_void_p), ("ev_c", C.c_void_p), ("esc", C.c_void_p)]


class COutboxC(C.Structure):
    _fields_ = [("plan_c", C.c_void_p), ("rep_c", C.c_void_p),
                ("commit_index", C.c_void_p), ("current_term", C.c_void_p), ("role_word", C.c_void_p), ("incarnation", C.c_void_p),
                ("err_word", C.c_void_p), ("last_entry", C.c_void_p), ("epoch", C.c_void_p), ("esc", C.c_void_p),
                ("esc_cap", C.c_uint32), ("_pad", C.c_uint32), ("counts", C.c_void_p)]
