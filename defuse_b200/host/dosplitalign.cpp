// dosplitalign -- drop-in for the reference tool of the same name (tools/dosplitalign.cpp):
//   dosplitalign -f ref.fa -e exons.regions -u <frag mean> -s <frag sd> -n <minread> -x <maxread>
//                -r clusters.regions -i improper.sam -1 reads.1.fastq -2 reads.2.fastq -a out.alignments
// Same flags, inputs, candidate enumeration ORDER and output bytes as the reference built against
// libstdc++ (SURVEY.md 8c): the containers whose iteration order decides the record order
// (unordered_map<int,task>, unordered_set<string> of transcripts, unordered_set<int> of overlapping
// cluster ends) are the same std containers filled by the same sequence of inserts.
// SplitReadAligner::Align + GetAlignments (tools/SplitAlignment.cpp:376-379) run on the GPU through
// dfb_split_align_batch; de-duplication and min(score1,score2) (:381-400) stay on the host.
//
// Built with -DDFB_FUSED_EVAL the same source is dosplitalign_eval, the fused align -> evaluate tool (SURVEY.md 8f rank 2):
//   dosplitalign_eval <the flags above, -a optional> -q out.seq -b out.break -p out.predalign
// The records stay in memory, are put into the order the pipeline's `sort -n -k 1` gives the alignments file
// (scripts/defuse_run.pl:528,533: numeric on the fusion id, whole line bytewise among equals, C locale) and go straight
// into evalsplitalign's evaluation (eval_core.h): the three outputs are byte-identical to
// dosplitalign | sort | evalsplitalign, without the multi-gigabyte intermediate file, the sort and the second parse.
// One process must see every read of the fusions it evaluates (one fastq split, or all of them).
//
// Built with -DDFB_MULTI_SPLIT it is dosplitalign_multi, every fastq split of a run in one process:
//   dosplitalign_multi -f ref.fa -e exons.regions -u <mean> -s <sd> -n <minread> -x <maxread> -r clusters.regions -l splits.tsv
// where each line of splits.tsv is "seq1.fastq <TAB> seq2.fastq <TAB> improper.sam <TAB> out.alignments".  Files,
// stdout, stderr and exit code are those of the stock tool run once per line, in order, stopping at the first run that
// fails; the set-up every split shares (regions, reference, exons, tasks, window table, bins, GPU contexts) is done once.
#if defined(DFB_FUSED_EVAL) && defined(DFB_MULTI_SPLIT)
#error "dosplitalign_eval and dosplitalign_multi are separate tools"
#endif
#include "split_tasks.h"
#include "fast_io.h"
#ifdef DFB_FUSED_EVAL
#include "eval_core.h"
#endif

#include <algorithm>
#include <fstream>
#include <map>
#include <memory>
#include <set>
#include <thread>
#include <unordered_map>
#include <unordered_set>

using namespace dfbhost;

namespace
{
struct Candidate
{
	int cluster_id; // fusion id
	int read_id;    // PackId(fragment, end) of the read to align (the OTHER end of the SAM record's fragment)
	int rev_comp;
};

#ifdef DFB_FUSED_EVAL
// `sort -n -k 1` in the C locale over the lines of `text`: by leading integer, lines with equal numbers bytewise
// (sort's last-resort comparison).  Counting sort on the fusion id, the lines of a fusion ordered by one thread.
std::string SortRecordsLikeThePipeline(const std::string& text)
{
	struct Line
	{
		const char* b;
		uint32_t len; // without the newline
		int id;
	};
	std::vector<Line> lines;
	for (const char *a = text.data(), *end = a + text.size(); a < end;)
	{
		const char* nl = (const char*)memchr(a, '\n', (size_t)(end - a));
		const char* e = nl ? nl : end;
		int id = 0;
		const char* t = (const char*)memchr(a, '\t', (size_t)(e - a));
		ParseIntRange(a, t ? t : e, id);
		lines.push_back(Line{a, (uint32_t)(e - a), id});
		a = nl ? nl + 1 : end;
	}
	std::vector<int> ids;
	ids.reserve(lines.size());
	for (const Line& l : lines) ids.push_back(l.id);
	std::sort(ids.begin(), ids.end());
	ids.erase(std::unique(ids.begin(), ids.end()), ids.end());
	std::vector<size_t> begin(ids.size() + 1, 0);
	std::vector<uint32_t> rank(lines.size());
	for (size_t k = 0; k < lines.size(); k++)
	{
		rank[k] = (uint32_t)(std::lower_bound(ids.begin(), ids.end(), lines[k].id) - ids.begin());
		begin[rank[k] + 1]++;
	}
	for (size_t k = 0; k < ids.size(); k++) begin[k + 1] += begin[k];
	std::vector<Line> sorted(lines.size());
	{
		std::vector<size_t> at(begin.begin(), begin.end() - 1);
		for (size_t k = 0; k < lines.size(); k++) sorted[at[rank[k]]++] = lines[k];
	}
	const int T = ToolThreads();
	ParallelRun(T, [&](int tid) {
		for (size_t f = (size_t)tid; f < ids.size(); f += (size_t)T)
			std::sort(sorted.begin() + (ptrdiff_t)begin[f], sorted.begin() + (ptrdiff_t)begin[f + 1], [](const Line& x, const Line& y) {
				const int c = memcmp(x.b, y.b, std::min(x.len, y.len));
				return c != 0 ? c < 0 : x.len < y.len;
			});
	});
	std::string out;
	out.reserve(text.size() + 1);
	for (const Line& l : sorted)
	{
		out.append(l.b, l.len);
		out += '\n';
	}
	return out;
}
#endif

// Where a split's messages go: straight to the streams, or -- for a split whose ingest runs while the split before it
// is still being aligned and written -- held until Release(), which writes them in the order they were said.
class Messages
{
public:
	explicit Messages(bool hold) : mHold(hold) {}
	void Out(const std::string& s) { Say(&std::cout, s); }
	void Err(const std::string& s) { Say(&std::cerr, s); }
	void Release()
	{
		for (const auto& m : mHeld) *m.first << m.second << std::flush;
		mHeld.clear();
	}

private:
	void Say(std::ostream* stream, const std::string& s)
	{
		if (s.empty()) return;
		if (mHold) mHeld.emplace_back(stream, s);
		else *stream << s << std::flush;
	}
	bool mHold;
	std::vector<std::pair<std::ostream*, std::string>> mHeld;
};

// What every split reads and nothing changes after the set-up: the GPU contexts, the tasks, the window table (window
// pair 2k, 2k+1 of cluster slot k) and the 2 000-bp bins of the mate regions.
struct SharedSetup
{
	std::vector<std::unique_ptr<Gpu>> gpus;
	std::unordered_map<int, ClusterTask> tasks; // its iteration order is the order mate regions are registered in
	BinnedRegions binned{2000};
	std::unordered_map<int, int> cluster_slot; // fusion id -> dense index (window pair 2k, 2k+1)
	TableBuilder windows;
};

void ReadSharedSetup(const CommandLine& cmd, SharedSetup& s, PhaseTimer& timer)
{
	// one context per GPU (DFB_DEVICES), created in the background while the inputs are parsed; candidates are
	// dealt out by cluster, no exchange between GPUs
	for (int dev : DeviceList()) s.gpus.emplace_back(new Gpu(dev));
	const double frag_mean = cmd.Double('u', 0.0), frag_sd = cmd.Double('s', 0.0);
	const int min_read = cmd.Int('n'), max_read = cmd.Int('x');

	// ---- clusters -> tasks (tools/dosplitalign.cpp:80-91, SplitAlignment.cpp:657-686) ----
	std::map<int, std::vector<Location>> regions;
	ReadRegionPairs(cmd.Str('r'), regions);
	FastaIndex reference;
	reference.Open(cmd.Str('f'));
	ExonModel exons;
	{
		std::ifstream in(cmd.Str('e').c_str());
		if (!in.good() || !exons.Read(in))
		{
			std::cerr << "Error: Unable to read exon regions file " << cmd.Str('e') << std::endl;
			ExitNow(1);
		}
	}
	for (const auto& kv : regions)
		InitializeTask(s.tasks[kv.first], kv.first, kv.second, reference, exons, frag_mean, frag_sd, min_read, max_read);

	timer.Lap("regions, fasta, exons, tasks");
	for (const auto& kv : s.tasks)
	{
		const ClusterTask& t = kv.second;
		s.cluster_slot[t.fusion_id] = (int)(s.windows.Count() / 2);
		s.windows.Add(t.window[0]);
		s.windows.Add(t.window[1]);
		for (int end = 0; end <= 1; end++)
			for (const Location& loc : t.mate_regions[end]) s.binned.Add(PackId(t.fusion_id, end), loc);
	}
	timer.Lap("bins");
}

// the four paths of one split (`write_align` false: dosplitalign_eval without -a)
struct SplitPaths
{
	std::string seq1, seq2, improper, align;
	bool write_align = true;
};

// what a split's ingest leaves for its alignment: both fastq files indexed in place, the candidates in order
struct SplitInput
{
	FastqIndex fastq[2];
	std::unique_ptr<Candidate[]> candidates;
	size_t n_candidates = 0;
};

// Host buffers of the batches, kept from batch to batch and from split to split.
struct Shard
{
	// the batch's reads as a CSR table; the bytes are a plain array that the worker threads touch first
	std::unique_ptr<char[]> read_bytes;
	size_t read_bytes_cap = 0;
	std::vector<int64_t> read_off;
	std::vector<int32_t> task_cluster, task_read, task_min_score, best, read_len, ref2_len;
	std::vector<int64_t> row_begin; // first result row of each task (n_rows when it has none)
	const dfb_split_row* rows = nullptr;
	const int32_t* cols = nullptr;
	int64_t n_rows = 0, n_cols = 0;
	int rc = DFB_OK;
};
struct BatchBuffers
{
	explicit BatchBuffers(int n_gpus) : shards((size_t)n_gpus), out_parts((size_t)ToolThreads()) {}
	std::vector<Shard> shards;
	std::vector<int> gpu_of;
	std::vector<int32_t> local_of;        // index of a candidate inside its shard
	std::vector<const char*> cand_seq;    // the candidate's read in the mapped fastq (forward orientation)
	std::vector<uint32_t> cand_len;
	std::vector<int32_t> cand_slot;
	std::vector<std::string> out_parts;
};

// One split up to its candidates: FASTQ index, SAM parse, overlaps, de-duplication.  false: the split fails here, its
// messages said (the stock tool exits 1 at that point).
bool IngestSplit(const SharedSetup& s, const SplitPaths& paths, SplitInput& in, Messages& msg, PhaseTimer& timer)
{
	// ---- reads: both fastq files indexed in place on a helper thread while the SAM file is parsed ----
	FastqIndex* const fastq = in.fastq;
	const bool ok0 = fastq[0].Open(paths.seq1);
	const bool ok1 = fastq[1].Open(paths.seq2);
	msg.Err(fastq[0].Message() + fastq[1].Message());
	if (!ok0 || !ok1)
	{
		msg.Out("Error: unable to read sequences\n");
		return false;
	}
	const int T = ToolThreads();
	std::thread fastq_thread([&] {
		fastq[0].Scan(std::max(1, T / 2));
		fastq[1].Scan(std::max(1, T / 2));
	});

	// The reference reads both fastq files to the end before it opens the SAM file (tools/dosplitalign.cpp:93-110), so
	// whatever the fastq streams have to say -- and a fatal fragment name -- comes before any SAM error.
	auto finish_fastq = [&]() {
		if (!fastq_thread.joinable()) return true;
		fastq_thread.join();
		for (int file = 0; file <= 1; file++)
		{
			msg.Err(fastq[file].Message());
			if (fastq[file].Fatal()) return false;
		}
		return true;
	};

	timer.Lap("fastq open");

	// ---- candidates, in the reference's order (SplitAlignment.cpp:266-303): SAM record order x iteration order of
	//      the overlap set; once per (cluster, read id, revComp).  Chunks of lines are parsed in parallel (every chunk
	//      keeps, per record, the overlap set in its iteration order), then merged in file order. ----
	// (plain arrays below: a std::vector would zero hundreds of megabytes on one thread before the workers fill them)
	std::unique_ptr<Candidate[]>& candidates = in.candidates;
	size_t& n_candidates = in.n_candidates;
	{
		MappedInput sam;
		const bool opened = paths.improper == "-" ? sam.OpenStdin() : sam.OpenFile(paths.improper);
		if (!opened)
		{
			if (!finish_fastq()) return false;
			msg.Err("Error: Unable to open sam file " + paths.improper + "\n");
			return false;
		}
		const char* const base = sam.data();
		std::vector<LineChunk> chunks = SplitLines(base, sam.size(), T);
		struct Part
		{
			std::vector<int32_t> stream; // per record with overlaps: fragment index, read end of the record, k, k ids
			int64_t error_line = -1;     // first fatal line of the chunk (1-based, global)
			std::string error;
		};
		std::vector<Part> parts(chunks.size());
		ParallelRun((int)chunks.size(), [&](int c) {
			Part& part = parts[(size_t)c];
			const char* a = base + chunks[(size_t)c].begin;
			const char* const end = base + chunks[(size_t)c].end;
			int64_t line_number = chunks[(size_t)c].first_line;
			std::string ref_name;
			auto fail = [&](const std::string& what) {
				part.error_line = line_number;
				part.error = what;
			};
			while (a < end)
			{
				const char* nl = (const char*)memchr(a, '\n', (size_t)(end - a));
				const char* const b = a;
				const char* const e = nl ? nl : end;
				a = nl ? nl + 1 : end;
				line_number++;
				if (b == e) return fail("Error: Empty alignment line " + std::to_string(line_number));
				if (*b == '@') continue;
				const char* f[11]; // starts of fields 0..9, f[10] = one past field 9
				int nf = 0;
				f[0] = b;
				for (const char* q = b; nf < 10;)
				{
					const char* t = (const char*)memchr(q, '\t', (size_t)(e - q));
					if (!t)
					{
						if (nf == 9) f[++nf] = e + 1;
						break;
					}
					f[++nf] = t + 1;
					q = t + 1;
				}
				if (nf < 10) return fail("Error: Format error for alignment line " + std::to_string(line_number));
				int flag = 0, pos = 0;
				if (!ParseIntRange(f[1], f[2] - 1, flag)) return fail("Error: bad lexical cast: flag '" + std::string(f[1], f[2] - 1) + "'");
				if (!ParseIntRange(f[3], f[4] - 1, pos)) return fail("Error: bad lexical cast: pos '" + std::string(f[3], f[4] - 1) + "'");
				if (f[3] - 1 - f[2] == 1 && *f[2] == '*') continue;
				const int strand = (flag & 0x0010) == 0 ? kPlus : kMinus;
				const char* const qb = f[0];
				const char* const qe = f[1] - 1;
				const char* slash = (const char*)memchr(qb, '/', (size_t)(qe - qb));
				const bool one_slash = slash && !memchr(slash + 1, '/', (size_t)(qe - slash - 1));
				const char* fragment_end = qe;
				int read_end = 0;
				if (one_slash)
				{
					if (qe - slash != 2 || (slash[1] != '1' && slash[1] != '2'))
						return fail("Error: Unable to interpret qname for alignment line " + std::to_string(line_number));
					fragment_end = slash;
					read_end = slash[1] == '1' ? 0 : 1;
				}
				else
				{
					if (flag & 0x0040) read_end = 0;
					else if (flag & 0x0080) read_end = 1;
					// (neither flag: the reference leaves readEnd uninitialised, AlignmentStream.cpp:108-116; end 0 here)
				}
				const Region r{pos, pos + (int)(f[10] - 1 - f[9]) - 1};
				ref_name.assign(f[2], f[3] - 1);
				std::unordered_set<int> overlapping;
				s.binned.Overlapping(ref_name, strand, r, overlapping);
				if (overlapping.empty()) continue;
				int fragment_index = 0;
				if (!ParseIntRange(qb, fragment_end, fragment_index))
					return fail("Error: bad lexical cast: fragment index '" + std::string(qb, fragment_end) + "'");
				part.stream.push_back(fragment_index);
				part.stream.push_back(read_end);
				part.stream.push_back((int32_t)overlapping.size());
				for (int cluster_end_id : overlapping) part.stream.push_back(cluster_end_id);
			}
		});
		for (const Part& part : parts)
			if (part.error_line >= 0)
			{
				// (chunks are in file order: this is the first line a sequential reader would have died on)
				if (!finish_fastq()) return false;
				msg.Err(part.error + "\n");
				return false;
			}
		timer.Lap("sam parse + overlaps");
		// expand the per-chunk streams into one candidate list (file order), then keep the first occurrence of every
		// (cluster, read id, revComp): the keys are dealt out to threads by hash, every thread walks the list in order
		// and decides the keys it owns
		std::vector<size_t> part_base(parts.size() + 1, 0);
		for (size_t c = 0; c < parts.size(); c++)
		{
			size_t m = 0;
			const std::vector<int32_t>& st = parts[c].stream;
			for (size_t q = 0; q < st.size(); q += 3 + (size_t)st[q + 2]) m += (size_t)st[q + 2];
			part_base[c + 1] = part_base[c] + m;
		}
		const size_t total = part_base.back();
		std::unique_ptr<uint64_t[]> keys(new uint64_t[total + 1]); // key = cluster id, read id, revComp: the whole candidate
		ParallelRun((int)parts.size(), [&](int c) {
			const std::vector<int32_t>& st = parts[(size_t)c].stream;
			size_t at = part_base[(size_t)c];
			for (size_t q = 0; q < st.size();)
			{
				const int fragment_index = st[q], read_end = st[q + 1], k = st[q + 2];
				q += 3;
				for (int j = 0; j < k; j++, q++, at++)
				{
					const int cluster_id = IdIndex(st[q]), cluster_end = IdEnd(st[q]);
					const int read_id = PackId(fragment_index, read_end == 0 ? 1 : 0);
					const int rev_comp = cluster_end == 0 ? 1 : 0;
					keys[at] = ((uint64_t)(uint32_t)cluster_id << 33) | ((uint64_t)(uint32_t)read_id << 1) | (uint64_t)rev_comp;
				}
			}
		});
		parts.clear();
		// first occurrence of every key, in list order: the positions are dealt into P buckets by key hash (a stable
		// counting sort: ranges of the list are scanned in parallel and write behind one another), every bucket is
		// then resolved by one thread with its own set, and the survivors are compacted range by range
		std::vector<uint8_t> keep(total, 0);
		const int P = total < (getenv("DFB_TOOL_CHUNK_MIN") ? (size_t)64 : (size_t)100000) ? 1 : T; // (tests shrink the chunks and this with them)
		if (P == 1)
		{
			KeySet seen(total + 16);
			for (size_t k = 0; k < total; k++)
				if (seen.Insert(keys[k])) keep[k] = 1;
		}
		else
		{
			// (many more buckets than threads: a bucket's set then fits the cache of the core that resolves it)
			int log_b = 1;
			while ((1 << log_b) < P || (log_b < 10 && (total >> log_b) > 32768)) log_b++;
			const int B = 1 << log_b;
			auto bucket_of = [log_b](uint64_t key) { return (int)((key * 0xD6E8FEB86659FD93ull) >> (64 - log_b)); };
			std::vector<size_t> count((size_t)P * (size_t)B, 0); // [range][bucket]
			ParallelRun(P, [&](int r) {
				size_t* cnt = &count[(size_t)r * (size_t)B];
				for (size_t k = total * (size_t)r / (size_t)P; k < total * ((size_t)r + 1) / (size_t)P; k++) cnt[bucket_of(keys[k])]++;
			});
			// bucket b holds [bucket_begin[b], bucket_begin[b+1]) of `order`; range r writes its part of b at start[r][b]
			std::vector<size_t> bucket_begin((size_t)B + 1, 0), start((size_t)P * (size_t)B, 0);
			for (int b = 0; b < B; b++)
			{
				size_t at = bucket_begin[(size_t)b];
				for (int r = 0; r < P; r++)
				{
					start[(size_t)r * (size_t)B + (size_t)b] = at;
					at += count[(size_t)r * (size_t)B + (size_t)b];
				}
				bucket_begin[(size_t)b + 1] = at;
			}
			const bool wide = total > 0xFFFFFFFFull;
			std::unique_ptr<uint32_t[]> order32(wide ? nullptr : new uint32_t[total + 1]);
			std::unique_ptr<uint64_t[]> order64(wide ? new uint64_t[total + 1] : nullptr);
			ParallelRun(P, [&](int r) {
				size_t* at = &start[(size_t)r * (size_t)B];
				for (size_t k = total * (size_t)r / (size_t)P; k < total * ((size_t)r + 1) / (size_t)P; k++)
				{
					const size_t pos = at[bucket_of(keys[k])]++;
					if (wide) order64[pos] = k; else order32[pos] = (uint32_t)k;
				}
			});
			ParallelRun(P, [&](int tid) {
				for (int b = tid; b < B; b += P)
				{
					const size_t lo = bucket_begin[(size_t)b], hi = bucket_begin[(size_t)b + 1];
					KeySet seen(hi - lo + 16);
					for (size_t q = lo; q < hi; q++)
					{
						const size_t k = wide ? (size_t)order64[q] : (size_t)order32[q];
						if (seen.Insert(keys[k])) keep[k] = 1;
					}
				}
			});
		}
		std::vector<size_t> kept_before((size_t)P + 1, 0);
		ParallelRun(P, [&](int r) {
			size_t c = 0;
			for (size_t k = total * (size_t)r / (size_t)P; k < total * ((size_t)r + 1) / (size_t)P; k++) c += keep[k];
			kept_before[(size_t)r + 1] = c;
		});
		for (int r = 0; r < P; r++) kept_before[(size_t)r + 1] += kept_before[(size_t)r];
		n_candidates = kept_before[(size_t)P];
		candidates.reset(new Candidate[n_candidates + 1]);
		ParallelRun(P, [&](int r) {
			size_t at = kept_before[(size_t)r];
			for (size_t k = total * (size_t)r / (size_t)P; k < total * ((size_t)r + 1) / (size_t)P; k++)
				if (keep[k])
					candidates[at++] = Candidate{(int)(uint32_t)(keys[k] >> 33), (int)(uint32_t)((keys[k] >> 1) & 0xFFFFFFFFull), (int)(keys[k] & 1)};
		});
	}
	timer.Lap("candidates (dedupe)");
	if (!finish_fastq()) return false;
	timer.Lap("fastq (wait)");
	return true;
}

// One split from its candidates to its finished alignments file; `records` (the fused tool) also gets every record.
// false: the output cannot be opened, the message said.  A GPU that fails ends the process here, as in the stock tool;
// every split before this one is finished by then.
bool AlignSplit(const SharedSetup& s, const SplitPaths& paths, const SplitInput& in, BatchBuffers& buf, Messages& msg,
                PhaseTimer& timer, std::string* records)
{
	// ---- the reads the candidates need (the reference keeps every read of both files, SplitAlignment.cpp:253-264, the
	//      second file overwriting the first; a read id that is absent aligns as the empty string, :286) ----
	const FastqIndex* const fastq = in.fastq;
	auto find_read = [&](int id, const char*& seq, uint32_t& len) {
		if (fastq[1].Find(id, seq, len) || fastq[0].Find(id, seq, len)) return;
		seq = nullptr;
		len = 0;
	};
	const Candidate* const candidates = in.candidates.get();
	const size_t n_candidates = in.n_candidates;
	const std::vector<std::unique_ptr<Gpu>>& gpus = s.gpus;
	const int n_gpus = (int)gpus.size();
	const std::unordered_map<int, int>& cluster_slot = s.cluster_slot;
	const TableBuilder& windows = s.windows;
	const int T = ToolThreads();

	const bool write_align = paths.write_align;
	std::ofstream out;
	if (write_align) out.open(paths.align.c_str());
	if (write_align && !out.good())
	{
		msg.Err("Error: Unable to open " + paths.align + "\n");
		return false;
	}

	// ---- align in batches, write records in candidate order ----
	const dfb_split_params params{kMatch, kMismatch, kGap, 0, kMinAnchor * kMatch};
	const dfb_seq_table window_table = windows.View();
	size_t kBatch = (size_t)(1u << 20) * (size_t)n_gpus; // (a batch twice as large costs the process another ~0.4 s of first-use device allocation)
	if (const char* e = getenv("DFB_TOOL_BATCH")) kBatch = (size_t)std::max(1, atoi(e)); // tests: force several batches
	std::vector<Shard>& shards = buf.shards;
	std::vector<int>& gpu_of = buf.gpu_of;
	std::vector<int32_t>& local_of = buf.local_of;
	std::vector<const char*>& cand_seq = buf.cand_seq;
	std::vector<uint32_t>& cand_len = buf.cand_len;
	std::vector<int32_t>& cand_slot = buf.cand_slot;
	std::vector<std::string>& out_parts = buf.out_parts;
	timer.Lap("open output");
	static unsigned char complement[256];
	for (int k = 0; k < 256; k++) complement[k] = (unsigned char)k;
	for (int k = 0; k < 8; k++) complement[(unsigned char)"ACGTacgt"[k]] = (unsigned char)"TGCAtgca"[k]; // tools/Common.cpp:32-54
	for (size_t first = 0; first < n_candidates; first += kBatch)
	{
		const size_t last = std::min(n_candidates, first + kBatch);
		const size_t n = last - first;
		cand_seq.resize(n);
		cand_len.resize(n);
		cand_slot.resize(n);
		ParallelRun(T, [&](int tid) {
			for (size_t k = n * (size_t)tid / (size_t)T; k < n * ((size_t)tid + 1) / (size_t)T; k++)
			{
				const Candidate& c = candidates[first + k];
				find_read(c.read_id, cand_seq[k], cand_len[k]);
				cand_slot[k] = cluster_slot.find(c.cluster_id)->second;
			}
		});
		timer.Add("batch: read lookup");
		// partition by cluster, heaviest first onto the lightest GPU (cost = DP cells); a cluster heavier than a
		// quarter of the mean load is cut into runs of candidates (every GPU holds every window pair)
		gpu_of.assign(n, 0);
		if (n_gpus > 1)
		{
			struct Unit
			{
				double cost;
				std::vector<int32_t> members;
			};
			std::unordered_map<int, std::vector<int32_t>> by_cluster;
			std::vector<int> cluster_order;
			std::vector<double> cost(n);
			double total = 0;
			for (size_t k = 0; k < n; k++)
			{
				const int slot = cand_slot[k];
				cost[k] = (double)cand_len[k] * (double)(windows.off[2 * slot + 2] - windows.off[2 * slot]);
				total += cost[k];
				auto ins = by_cluster.emplace(candidates[first + k].cluster_id, std::vector<int32_t>());
				if (ins.second) cluster_order.push_back(candidates[first + k].cluster_id);
				ins.first->second.push_back((int32_t)k);
			}
			const double cap = std::max(1.0, total / n_gpus / 4.0);
			std::vector<Unit> units;
			for (int cid : cluster_order)
			{
				Unit u{0.0, {}};
				for (int32_t k : by_cluster[cid])
				{
					if (u.cost > cap)
					{
						units.push_back(std::move(u));
						u = Unit{0.0, {}};
					}
					u.members.push_back(k);
					u.cost += cost[k];
				}
				if (!u.members.empty()) units.push_back(std::move(u));
			}
			std::stable_sort(units.begin(), units.end(), [](const Unit& a, const Unit& b) { return a.cost > b.cost; });
			std::vector<double> load((size_t)n_gpus, 0.0);
			for (const Unit& u : units)
			{
				const int g = (int)(std::min_element(load.begin(), load.end()) - load.begin());
				load[g] += u.cost;
				for (int32_t k : u.members) gpu_of[k] = g;
			}
		}
		// shard tables: offsets by one sequential pass over arrays that keep their size from batch to batch (nothing is
		// re-zeroed: every entry in use is written below), bytes (reverse-complemented where the candidate says so) in
		// parallel
		local_of.resize(n);
		std::vector<size_t> shard_tasks((size_t)n_gpus, 0);
		for (Shard& sh : shards)
		{
			if (sh.task_cluster.size() < n) sh.task_cluster.resize(n);
			if (sh.read_off.size() < n + 1) sh.read_off.resize(n + 1);
			sh.read_off[0] = 0;
		}
		if (n_gpus == 1)
		{
			// one shard: task k is candidate k, offsets are a prefix sum over ranges of candidates
			Shard& sh = shards[0];
			std::vector<int64_t> range_bytes((size_t)T + 1, 0);
			ParallelRun(T, [&](int tid) {
				int64_t sum = 0;
				for (size_t k = n * (size_t)tid / (size_t)T; k < n * ((size_t)tid + 1) / (size_t)T; k++) sum += (int64_t)cand_len[k];
				range_bytes[(size_t)tid + 1] = sum;
			});
			for (int r = 0; r < T; r++) range_bytes[(size_t)r + 1] += range_bytes[(size_t)r];
			ParallelRun(T, [&](int tid) {
				int64_t at = range_bytes[(size_t)tid];
				for (size_t k = n * (size_t)tid / (size_t)T; k < n * ((size_t)tid + 1) / (size_t)T; k++)
				{
					local_of[k] = (int32_t)k;
					sh.task_cluster[k] = cand_slot[k];
					at += (int64_t)cand_len[k];
					sh.read_off[k + 1] = at;
				}
			});
			shard_tasks[0] = n;
		}
		else
		{
			for (size_t k = 0; k < n; k++)
			{
				const int g = gpu_of[k];
				Shard& sh = shards[(size_t)g];
				const size_t t = shard_tasks[(size_t)g]++;
				local_of[k] = (int32_t)t;
				sh.task_cluster[t] = cand_slot[k];
				sh.read_off[t + 1] = sh.read_off[t] + (int64_t)cand_len[k];
			}
		}
		for (int g = 0; g < n_gpus; g++)
		{
			Shard& sh = shards[(size_t)g];
			const size_t m = shard_tasks[(size_t)g];
			sh.task_cluster.resize(m);
			sh.read_off.resize(m + 1);
			if (sh.read_bytes_cap < (size_t)sh.read_off[m] + 1)
			{
				sh.read_bytes_cap = (size_t)sh.read_off[m] + (size_t)sh.read_off[m] / 8 + 64;
				sh.read_bytes.reset(new char[sh.read_bytes_cap]);
			}
			sh.task_read.resize(m);
			sh.task_min_score.resize(m);
			sh.read_len.resize(m);
			sh.ref2_len.resize(m);
			sh.best.resize(m);
		}
		ParallelRun(T, [&](int tid) {
			for (size_t k = n * (size_t)tid / (size_t)T; k < n * ((size_t)tid + 1) / (size_t)T; k++)
			{
				Shard& sh = shards[gpu_of[k]];
				const int32_t t = local_of[k];
				const uint32_t len = cand_len[k];
				char* dst = sh.read_bytes.get() + sh.read_off[(size_t)t];
				const char* src = cand_seq[k];
				if (candidates[first + k].rev_comp)
					for (uint32_t q = 0; q < len; q++) dst[q] = (char)complement[(unsigned char)src[len - 1 - q]];
				else if (len)
					memcpy(dst, src, len);
				const int slot = cand_slot[k];
				sh.task_read[(size_t)t] = t;
				sh.task_min_score[(size_t)t] = (int)((float)len * (float)kMatch * 0.90); // SplitAlignment.cpp:379
				sh.read_len[(size_t)t] = (int32_t)len;
				sh.ref2_len[(size_t)t] = (int32_t)(windows.off[2 * slot + 2] - windows.off[2 * slot + 1]);
			}
		});
		timer.Add("batch: tables");
		for (auto& g : gpus) g->ctx();
		timer.Add("batch: wait for gpu context");
		auto run_shard = [&](int g) {
			Shard& sh = shards[g];
			const dfb_seq_table read_table{(const uint8_t*)sh.read_bytes.get(), sh.read_off.data(), (int64_t)sh.read_off.size() - 1};
			sh.rc = dfb_split_align_batch(gpus[g]->ctx(), &params, &window_table, &read_table, sh.task_cluster.data(),
			                              sh.task_read.data(), sh.task_min_score.data(), (int64_t)sh.task_cluster.size(),
			                              sh.best.data());
			if (sh.rc == DFB_OK) sh.rc = dfb_split_result_view(gpus[g]->ctx(), &sh.rows, &sh.n_rows, &sh.cols, &sh.n_cols);
			if (sh.rc != DFB_OK) return;
			if (n_gpus == 1) timer.Add("batch: gpu call");
			// rows come in task order: where each task's rows start
			sh.row_begin.assign(sh.task_cluster.size() + 1, sh.n_rows);
			for (int64_t r = sh.n_rows - 1; r >= 0; r--) sh.row_begin[(size_t)sh.rows[r].task] = r;
			for (int64_t t = (int64_t)sh.task_cluster.size() - 1; t >= 0; t--)
				if (sh.row_begin[(size_t)t] == sh.n_rows) sh.row_begin[(size_t)t] = sh.row_begin[(size_t)t + 1];
		};
		if (n_gpus == 1)
		{
			run_shard(0);
		}
		else
		{
			std::vector<std::thread> th;
			for (int g = 0; g < n_gpus; g++) th.emplace_back(run_shard, g);
			for (auto& t : th) t.join();
		}
		for (int g = 0; g < n_gpus; g++)
			if (shards[g].rc != DFB_OK) gpus[g]->Die("split alignment failed");

		timer.Add("batch: row index");
		// records of the candidates in their original order, formatted by ranges of candidates
		ParallelRun(T, [&](int tid) {
			std::string& os = out_parts[(size_t)tid];
			os.clear();
			std::vector<std::pair<int, int>> small; // refSplits of the task seen so far
			std::unordered_set<std::pair<int, int>, PairHash> large;
			for (size_t k = n * (size_t)tid / (size_t)T; k < n * ((size_t)tid + 1) / (size_t)T; k++)
			{
				const Shard& sh = shards[gpu_of[k]];
				const int32_t t = local_of[k];
				const int64_t r0 = sh.row_begin[(size_t)t], r1 = sh.row_begin[(size_t)t + 1];
				if (r0 == r1) continue;
				const Candidate& c = candidates[first + k];
				small.clear();
				large.clear();
				for (int64_t r = r0; r < r1; r++)
				{
					const dfb_split_row& row = sh.rows[r];
					const int32_t* c1 = sh.cols + row.col_begin;
					const int32_t* c2 = c1 + row.n1;
					const int score = std::min(row.score1, row.score2); // SplitAlignment.cpp:400
					for (int a = 0; a < row.n1; a++)
					{
						for (int b = 0; b < row.n2; b++)
						{
							const std::pair<int, int> ref_split(c1[a], sh.ref2_len[(size_t)t] - c2[b] - 1); // SplitReadAligner.cpp:277-278
							// first per refSplit (SplitAlignment.cpp:383-390)
							bool fresh;
							if (large.empty() && small.size() < 32)
							{
								fresh = std::find(small.begin(), small.end(), ref_split) == small.end();
								if (fresh) small.push_back(ref_split);
							}
							else
							{
								if (large.empty()) large.insert(small.begin(), small.end());
								fresh = large.insert(ref_split).second;
							}
							if (!fresh) continue;
							AppendInt(os, c.cluster_id);
							os += '\t';
							AppendInt(os, IdIndex(c.read_id));
							os += '\t';
							AppendInt(os, IdEnd(c.read_id));
							os += '\t';
							AppendInt(os, c.rev_comp);
							os += '\t';
							AppendInt(os, ref_split.first);
							os += '\t';
							AppendInt(os, ref_split.second);
							os += '\t';
							AppendInt(os, row.read_split);
							os += '\t';
							AppendInt(os, sh.read_len[(size_t)t] - row.read_split);
							os += '\t';
							AppendInt(os, score);
							os += "\t\n";
						}
					}
				}
			}
		});
		timer.Add("batch: format");
		if (write_align)
			for (const std::string& part : out_parts) out.write(part.data(), (std::streamsize)part.size());
		if (records)
			for (const std::string& part : out_parts) *records += part;
		timer.Add("batch: write");
	}
	if (write_align)
	{
		out.flush();
		out.close();
	}
	return true;
}

#ifdef DFB_MULTI_SPLIT
// The split manifest: one split per line, four TAB-separated paths (seq1.fastq, seq2.fastq, improper.sam, output).
// Anything malformed ends the run before a split is read or an output created.
std::vector<SplitPaths> ReadManifest(const std::string& path)
{
	auto fail = [](const std::string& what) {
		std::cerr << "Error: " << what << std::endl;
		ExitNow(1);
	};
	std::ifstream in(path.c_str());
	if (!in.good()) fail("Unable to read splits manifest " + path);
	std::vector<SplitPaths> splits;
	std::set<std::string> outputs;
	std::string line;
	std::vector<std::string> f;
	while (std::getline(in, line))
	{
		const std::string where = "splits manifest " + path + " line " + std::to_string(splits.size() + 1);
		SplitChar(line, '\t', f);
		if (f.size() != 4 || f[0].empty() || f[1].empty() || f[2].empty() || f[3].empty())
			fail("Expected four non-empty tab-separated fields (seq1, seq2, improper sam, output) on " + where);
		for (const std::string& p : f)
			if (p == "-") fail("'-' names standard input or output, which cannot serve several splits, on " + where);
		if (!outputs.insert(f[3]).second) fail("Output " + f[3] + " is named a second time on " + where);
		splits.push_back(SplitPaths{f[0], f[1], f[2], f[3]});
	}
	if (in.bad()) fail("Unable to read splits manifest " + path);
	if (splits.empty()) fail("Splits manifest " + path + " has no lines");
	return splits;
}
#endif

}  // namespace

#ifndef DFB_MULTI_SPLIT
int main(int argc, char* argv[])
{
	CommandLine cmd("Fusion sequence prediction by split reads", {
	    {'f', "fasta", "Reference Fasta", true, "string", "", false},
	    {'e', "exons", "Exon Regions Filename", true, "string", "", false},
	    {'u', "ufrag", "Fragment Length Mean", true, "float", "", false},
	    {'s', "sfrag", "Fragment Length Standard Deviation", true, "float", "", false},
	    {'n', "minread", "Minimum Read Length", true, "integer", "", false},
	    {'x', "maxread", "Maximum Read Length", true, "integer", "", false},
	    {'r', "regions", "Fusion Regions Filename", true, "string", "", false},
	    {'i', "improper", "Improper Alignments Sam Filename", true, "string", "", false},
	    {'1', "seq1", "End 1 Sequences", true, "string", "", false},
	    {'2', "seq2", "End 2 Sequences", true, "string", "", false},
#ifdef DFB_FUSED_EVAL
	    {'a', "align", "Split Alignments Filename (optional here)", false, "string", "", false},
	    {'q', "seq", "Sequences Filename", true, "string", "", false},
	    {'b', "break", "Break Positions Filename", true, "string", "", false},
	    {'p', "predalign", "Prediction Split Alignments Filename", true, "string", "", false},
#else
	    {'a', "align", "Split Alignments Filename", true, "string", "", false},
#endif
	});
	cmd.Parse(argc, argv);
	PhaseTimer timer;
	SharedSetup shared;
	ReadSharedSetup(cmd, shared, timer);
	SplitPaths paths{cmd.Str('1'), cmd.Str('2'), cmd.Str('i'), cmd.Str('a')};
	std::string* records = nullptr;
#ifdef DFB_FUSED_EVAL
	paths.write_align = cmd.IsSet('a');
	std::string fused_text; // every record of the run, in emission order
	records = &fused_text;
#endif
	Messages direct(false);
	SplitInput in;
	if (!IngestSplit(shared, paths, in, direct, timer)) ExitNow(1);
	BatchBuffers buf((int)shared.gpus.size());
	if (!AlignSplit(shared, paths, in, buf, direct, timer, records)) ExitNow(1);
#ifdef DFB_FUSED_EVAL
	{
		// align -> evaluate without the file in between (tools/evalsplitalign.cpp:96-114 on the sorted records)
		std::ofstream seq_file(cmd.Str('q').c_str()), break_file(cmd.Str('b').c_str()), pred_file(cmd.Str('p').c_str());
		for (const char f : {'q', 'b', 'p'})
			if (!(f == 'q' ? seq_file : (f == 'b' ? break_file : pred_file)).good())
			{
				std::cerr << "Error: Unable to open " << cmd.Str(f) << std::endl;
				ExitNow(1);
			}
		const std::string sorted = SortRecordsLikeThePipeline(fused_text);
		timer.Lap("fused: sort records");
		const bool ok = EvaluateSortedRecords(sorted.data(), sorted.data() + sorted.size(), shared.tasks, seq_file, break_file, pred_file);
		timer.Lap("fused: evaluate");
		if (!ok) ExitNow(1);
	}
#endif
	timer.Report();
	timer.Lap("close");
	FinishProcess(0);
}
#else
int main(int argc, char* argv[])
{
	CommandLine cmd("Fusion sequence prediction by split reads, every fastq split of a run in one process", {
	    {'f', "fasta", "Reference Fasta", true, "string", "", false},
	    {'e', "exons", "Exon Regions Filename", true, "string", "", false},
	    {'u', "ufrag", "Fragment Length Mean", true, "float", "", false},
	    {'s', "sfrag", "Fragment Length Standard Deviation", true, "float", "", false},
	    {'n', "minread", "Minimum Read Length", true, "integer", "", false},
	    {'x', "maxread", "Maximum Read Length", true, "integer", "", false},
	    {'r', "regions", "Fusion Regions Filename", true, "string", "", false},
	    {'l', "splits", "Splits Manifest Filename (per line: seq1 <TAB> seq2 <TAB> improper sam <TAB> alignments)", true, "string", "", false},
	});
	cmd.Parse(argc, argv);
	const std::vector<SplitPaths> splits = ReadManifest(cmd.Str('l'));
	PhaseTimer timer;
	SharedSetup shared;
	ReadSharedSetup(cmd, shared, timer); // (says nothing unless it fails, and then it exits: said once, as by the first stock run)
	BatchBuffers buf((int)shared.gpus.size());
	// Split k+1's ingest runs on a helper thread while split k is aligned and written, its messages held until split k
	// is done; at most two splits' inputs are mapped at once.  DFB_SPLIT_OVERLAP=0: one split after the other.
	const bool overlap = !(getenv("DFB_SPLIT_OVERLAP") && atoi(getenv("DFB_SPLIT_OVERLAP")) == 0);
	auto label = [](size_t k) { return "split " + std::to_string(k + 1) + ": "; };
	Messages direct(false);
	std::unique_ptr<SplitInput> current(new SplitInput);
	std::unique_ptr<PhaseTimer> split_timer(new PhaseTimer(label(0)));
	if (!IngestSplit(shared, splits[0], *current, direct, *split_timer)) ExitNow(1);
	for (size_t k = 0; k < splits.size(); k++)
	{
		const bool last = k + 1 == splits.size();
		std::unique_ptr<SplitInput> next;
		std::unique_ptr<PhaseTimer> next_timer;
		Messages held(true);
		bool next_ok = true;
		std::thread ahead;
		if (overlap && !last)
		{
			next.reset(new SplitInput);
			next_timer.reset(new PhaseTimer(label(k + 1)));
			ahead = std::thread([&] { next_ok = IngestSplit(shared, splits[k + 1], *next, held, *next_timer); });
		}
		split_timer->Restart();
		if (!AlignSplit(shared, splits[k], *current, buf, direct, *split_timer, nullptr)) ExitNow(1);
		split_timer->Report();
		current.reset(); // (split k's inputs are unmapped before split k+2's ingest maps more)
		if (last) break;
		if (overlap)
		{
			ahead.join();
			held.Release();
			if (!next_ok) ExitNow(1);
			current = std::move(next);
			split_timer = std::move(next_timer);
		}
		else
		{
			current.reset(new SplitInput);
			split_timer.reset(new PhaseTimer(label(k + 1)));
			if (!IngestSplit(shared, splits[k + 1], *current, direct, *split_timer)) ExitNow(1);
		}
	}
	timer.Lap("close");
	FinishProcess(0);
}
#endif
