"""CPU oracle (TEST INFRASTRUCTURE ONLY) for the unique-k-mer recruitment path.

A plain-Python restatement of the reference algorithm, in the reference's own
string domain, written as order-independent closed forms so that it can be
compared with the device path without depending on dict/set iteration order.
Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline
leg may import it; nothing under ``centroflye_b200/`` does.

Parity status: PINNED.  ``oracle/make_golden.py`` runs the unmodified reference
(/root/reference/scripts, with a stub ``Bio.SeqIO``) on seeded synthetic NCRF
reports and commits its outputs under ``tests/golden/``;
``tests/test_oracle_golden.py`` checks every function here against them.

Reference lines followed (relative to /root/reference/scripts):
  segment_units        ncrf_parser.py:28-59
  kmer_freqs           distance_based_kmer_recruitment.py:39-63
  rare_kmers           distance_based_kmer_recruitment.py:66-82
  reads_kmer_clouds    read_kmer_cloud.py:18-40
  filter_clouds        read_kmer_cloud.py:43-54
  dist_counts          distance_based_kmer_recruitment.py:85-128
  filter_edges         distance_based_kmer_recruitment.py:131-149
  result_files         distance_based_kmer_recruitment.py:152-171
  PlacerModel          read_placer.py:35-94 + cloud_contig.py:26-41,87-95, as centroflye_b200/read_placer.py
                       and csrc/placer.cu document them (checked against read_positions_<tag>.csv)
"""
import heapq
import itertools
import math
import re
from collections import Counter, defaultdict


def segment_units(r_al, m_al, motif, n=1):
    """[(start, end)] alignment-column intervals of the units (ncrf_parser.py:34-53)."""
    pattern = re.compile("".join(f"{b}-*" for b in motif) * n)
    matches = list(pattern.finditer(m_al.upper()))
    if not matches:
        return []
    coords = [m.start() for m in matches] + [matches[-1].end()]
    if coords[0] > len(motif) * 0.2:
        coords.insert(0, 0)
    if coords[-1] < len(r_al) - len(motif) * 0.2:
        coords.append(len(r_al))
    return list(zip(coords[:-1], coords[1:]))


def kmer_freqs(records, k, max_nonuniq):
    """kmer -> number of records containing it, for k-mers that occur more than once in at
    most ``max_nonuniq`` records.  Closed form of the sequential update at :55-62: the
    running ``non_unique_freqs`` only grows, so a k-mer survives iff its FINAL value is
    <= max_nonuniq, and while it survives every containing record adds one."""
    n_reads, n_multi = Counter(), Counter()
    for rec in records.values():
        s = rec.r_al.replace("-", "")
        per_read = Counter(s[i:i + k] for i in range(len(s) - k + 1))
        for kmer, c in per_read.items():
            n_reads[kmer] += 1
            if c > 1:
                n_multi[kmer] += 1
    return {kmer: c for kmer, c in n_reads.items() if n_multi[kmer] <= max_nonuniq}


def rare_band(bottom, top, coverage, kmer_survival_rate):
    # same evaluation order as :74-75 (float64)
    return bottom * coverage * kmer_survival_rate, top * coverage * kmer_survival_rate


def rare_kmers(records, k, bottom, top, coverage, kmer_survival_rate, max_nonuniq):
    left, right = rare_band(bottom, top, coverage, kmer_survival_rate)
    return {kmer for kmer, f in kmer_freqs(records, k, max_nonuniq).items() if left <= f <= right}


def reads_kmer_clouds(records, n, k, genomic_kmers):
    """r_id -> list (one per unit) of sets of genomic k-mers lying wholly inside the unit."""
    out = {}
    for r_id, rec in records.items():
        clouds = []
        for st, en in segment_units(rec.r_al, rec.m_al, rec.motif, n=n):
            u = rec.r_al[st:en].upper().replace("-", "")
            clouds.append({u[i:i + k] for i in range(len(u) - k + 1) if u[i:i + k] in genomic_kmers})
        out[r_id] = clouds
    return out


def filter_clouds(clouds, min_mult=2, max_mult=math.inf):
    mult = Counter(kmer for cl in clouds.values() for unit in cl for kmer in unit)
    return {r_id: [{kmer for kmer in unit if max_mult >= mult[kmer] >= min_mult} for unit in cl]
            for r_id, cl in clouds.items()}


def dist_counts(clouds, min_n, max_n, min_d, max_d):
    """(a, b, d) -> count over reads [min_n, max_n) of unit pairs (i, i+d) with a in unit i,
    b in unit i+d, a != b.  ``kmer_clouds[:-dist]`` at :121 makes dist = 0 contribute nothing."""
    cnt = defaultdict(int)
    for _, units in itertools.islice(clouds.items(), min_n, max_n):
        for d in range(max(min_d, 1), max_d + 1):
            for i in range(len(units) - d):
                for a in units[i]:
                    for b in units[i + d]:
                        if a != b:
                            cnt[(a, b, d)] += 1
    return cnt


def filter_edges(cnt, min_coverage, rel_threshold=0.8):
    total = defaultdict(int)
    for (a, b, _), c in cnt.items():
        total[(a, b)] += c
    edges = {(d, a, b, c) for (a, b, d), c in cnt.items()
             if c >= min_coverage and c / total[(a, b)] >= rel_threshold}
    selected = {e[1] for e in edges} | {e[2] for e in edges}
    return selected, edges


def recruit(records, k=19, coverage=32, min_coverage=4, min_n=0, max_n=None, min_d=1, max_d=150,
            bottom=0.9, top=3.0, kmer_survival_rate=0.34, max_nonuniq=3):
    """main() of the reference script, :174-208, returning everything along the way."""
    rare = rare_kmers(records, k, bottom, top, coverage, kmer_survival_rate, max_nonuniq)
    clouds = reads_kmer_clouds(records, 1, k, rare)
    cnt = dist_counts(clouds, min_n, max_n, min_d, max_d)
    selected, edges = filter_edges(cnt, min_coverage)
    return {"rare": rare, "clouds": clouds, "n_increments": sum(cnt.values()), "n_keys": len(cnt),
            "selected": selected, "edges": edges}


def result_files(selected, edges):
    """Contents of the two output files (:158-171) with the hash-seed dependent edge order
    canonicalised by sorting the lines."""
    kmers_txt = "".join(kmer + "\n" for kmer in sorted(selected))
    edge_lines = sorted(f"{d} {a} {b} {c}\n" for d, a, b, c in edges)
    return kmers_txt, edge_lines


class PlacerContig:
    """cloud_contig.CloudContig as the placer uses it: (position, k-mer) counters, every position each k-mer was
    added at, and the k-mers that reached min_cloud_kmer_freq at some position (0 counts as 1)."""

    def __init__(self, min_cloud_kmer_freq):
        self.min_freq = max(1, min_cloud_kmer_freq)
        self.cnt = Counter()                # (position, kmer) -> count
        self.positions = defaultdict(set)   # kmer -> positions it was added at
        self.freq = set()
        self.read_positions = {}
        self.coverage = defaultdict(int)
        self.max_pos = 0
        self._last = -1                     # last position any unit was added at

    def add_read(self, clouds, r_id, position):
        """Adds one read; returns the (kmer, position) pairs whose count reached min_freq just now."""
        self.read_positions[r_id] = position
        new = []
        for i, cloud in enumerate(clouds):
            p = position + i
            self.coverage[p] += 1
            for kmer in cloud:
                self.cnt[(p, kmer)] += 1
                self.positions[kmer].add(p)
                if self.cnt[(p, kmer)] == self.min_freq:
                    self.freq.add(kmer)
                    new.append((kmer, p))
        if len(clouds):
            self._last = max(self._last, position + len(clouds) - 1)
        self.max_pos = max(self._last, 0)
        return new


class PlacerModel:
    """ReadPlacer's greedy loop over plain dicts and sets of k-mer strings.  ``clouds`` maps r_id -> list of unit
    clouds.  ``lines`` is what read_positions.csv holds after the calls so far; ``decided`` counts, per pick, which
    level of the selection rule separated the winner from the best other candidate: "alone" (no other candidate),
    "score" (distinct positions, total), "offset" (the larger offset) or "r_id" (the smaller r_id string)."""

    def __init__(self, min_cloud_kmer_freq):
        self.contig = PlacerContig(min_cloud_kmer_freq)
        self.lines = []
        self.decided = Counter()
        self.scores = {}   # (r_id, offset) -> [distinct positions, total] of the last add_reads call

    def add_prefix_reads(self, prefix_reads, clouds):
        self.lines = []    # the file is rewritten
        for r_id in prefix_reads:
            self.contig.add_read(clouds[r_id], r_id, 0)
            self.lines.append(f"{r_id} 0")

    @staticmethod
    def _passes(distinct, total, min_unit, min_inters, min_prop):
        return distinct >= min_unit and total >= min_inters and total >= min_prop * distinct

    def add_reads(self, reads, clouds, min_unit, min_inters, min_prop=3):
        kmers2pos = defaultdict(list)
        for r_id in reads:
            for pos, cloud in enumerate(clouds[r_id]):
                for kmer in cloud:
                    kmers2pos[kmer].append((r_id, pos))
        seen = set()       # (r_id, offset, position in read)
        scores = self.scores = {}
        # candidates of unused reads, largest first; an entry is stale once its scores have moved on
        heap = []
        unused = set(reads)
        pairs = [(kmer, p) for kmer in self.contig.freq for p in self.contig.positions[kmer]]
        while unused:
            touched = set()
            for kmer, cc_pos in pairs:
                for r_id, pos in kmers2pos.get(kmer, ()):
                    if cc_pos < pos:
                        continue
                    off = cc_pos - pos
                    sc = scores.setdefault((r_id, off), [0, 0])
                    if (r_id, off, pos) not in seen:
                        seen.add((r_id, off, pos))
                        sc[0] += 1
                    sc[1] += 1
                    touched.add((r_id, off))
            for r_id, off in touched:
                d, t = scores[(r_id, off)]
                if r_id in unused and self._passes(d, t, min_unit, min_inters, min_prop):
                    heapq.heappush(heap, (-d, -t, -off, r_id))
            best = self._pop(heap, scores, unused)
            if best is None:
                self.lines += [f"{r_id} None" for r_id in reads if r_id in unused]
                return
            runner_up = self._pop(heap, scores, unused)
            if runner_up is None:
                self.decided["alone"] += 1
            else:
                heapq.heappush(heap, runner_up)
                level = "score" if runner_up[:2] != best[:2] else "offset" if runner_up[2] != best[2] else "r_id"
                self.decided[level] += 1
            d, t, off, r_id = -best[0], -best[1], -best[2], best[3]
            self.lines.append(f"{r_id} {off} {d} {t}")
            unused.discard(r_id)
            pairs = self.contig.add_read(clouds[r_id], r_id, off)

    @staticmethod
    def _pop(heap, scores, unused):
        while heap:
            e = heapq.heappop(heap)
            if e[3] in unused and scores[(e[3], -e[2])] == [-e[0], -e[1]]:
                return e
        return None


def place_reads(prefix, internal, suffix, clouds, min_cloud_kmer_freq, min_unit, min_inters, min_prop=3):
    """ReadPlacer.run after classification: prefix reads, then internal reads, then suffix reads."""
    model = PlacerModel(min_cloud_kmer_freq)
    model.add_prefix_reads(prefix, clouds)
    model.add_reads(internal, clouds, min_unit, min_inters, min_prop)
    model.add_reads(suffix, clouds, min_unit, min_inters, min_prop)
    return model
