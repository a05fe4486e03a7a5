// Shared host code of the three drop-in tools (localalign, matealign, dosplitalign).
// The tools keep the reference's command lines, input formats and output bytes; the DP itself
// goes through the C ABI (include/defuse_b200.h) in batches.  No CPU aligner exists here: if the
// library cannot create a context on a B200 the tool prints "Error: ..." and exits 1, which is how
// the reference tools report any failure (tools/DebugCheck.cpp:15-19) and what
// scripts/cmdrunner.pm:620-627 treats as a failed job.
#pragma once

#include "defuse_b200.h"

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <iostream>
#include <sstream>
#include <string>
#include <thread>
#include <unistd.h>
#include <vector>

namespace dfbhost
{
// Error exits of the tools: the reference calls exit(1) (tools/DebugCheck.cpp:15-19 and the I/O checks).  Here a GPU
// context may still be coming up on a helper thread, and exit() would run the CUDA runtime's teardown against it:
// flush what was written and leave at once.
[[noreturn]] inline void ExitNow(int code)
{
	std::cout.flush();
	std::cerr.flush();
	fflush(nullptr);
	_exit(code);
}


// ---------------------------------------------------------------------------------------------
// command line: the grammar the reference gets from TCLAP (include/tclap/CmdLine.h):
// "-f value" / "--name value", every listed argument takes one value, required-ness checked,
// "--" ends parsing, -h/--help and --version are built in; any error -> message on stderr, exit 1
// ---------------------------------------------------------------------------------------------
struct ArgSpec
{
	char flag;
	const char* name;
	const char* desc;
	bool required;
	const char* type_desc;
	std::string value;
	bool set;
};

class CommandLine
{
public:
	CommandLine(const char* prog_desc, std::vector<ArgSpec> specs) : mDesc(prog_desc), mSpecs(std::move(specs))
	{
		for (auto& s : mSpecs) s.set = false;
	}

	void Parse(int argc, char* argv[])
	{
		mProg = argc > 0 ? argv[0] : "tool";
		for (int i = 1; i < argc; i++)
		{
			std::string a = argv[i];
			if (a == "--") break; // TCLAP: ignore the rest
			if (a == "-h" || a == "--help")
			{
				Usage(std::cout, true);
				ExitNow(0);
			}
			if (a == "--version")
			{
				std::cout << std::endl << mProg << "  version: none" << std::endl << std::endl;
				ExitNow(0);
			}
			ArgSpec* spec = nullptr;
			if (a.size() == 2 && a[0] == '-' && a[1] != '-')
			{
				for (auto& s : mSpecs)
					if (s.flag == a[1]) spec = &s;
			}
			else if (a.size() > 2 && a[0] == '-' && a[1] == '-')
			{
				for (auto& s : mSpecs)
					if (a.substr(2) == s.name) spec = &s;
			}
			if (!spec) Fail("Argument: " + a, "Couldn't find match for argument");
			if (spec->set) Fail(ArgId(*spec), "Argument already set!");
			if (i + 1 >= argc) Fail(ArgId(*spec), "Missing a value for this argument!");
			spec->value = argv[++i];
			spec->set = true;
		}
		std::string missing;
		for (auto& s : mSpecs)
			if (s.required && !s.set) missing += (missing.empty() ? "" : ", ") + std::string(s.name);
		if (!missing.empty()) Fail("Required argument missing: " + missing, "One or more required arguments missing!");
	}

	bool IsSet(char flag) const { return Find(flag).set; }
	const std::string& Str(char flag) const { return Find(flag).value; }

	int Int(char flag) const
	{
		const ArgSpec& s = Find(flag);
		std::istringstream is(s.value);
		int v = 0;
		char extra;
		if (!(is >> v) || (is >> extra)) Fail(ArgId(s), "Couldn't read argument value from string '" + s.value + "'");
		return v;
	}

	double Double(char flag, double dflt) const
	{
		const ArgSpec& s = Find(flag);
		if (!s.set) return dflt;
		std::istringstream is(s.value);
		double v = 0;
		char extra;
		if (!(is >> v) || (is >> extra)) Fail(ArgId(s), "Couldn't read argument value from string '" + s.value + "'");
		return v;
	}

private:
	const ArgSpec& Find(char flag) const
	{
		for (auto& s : mSpecs)
			if (s.flag == flag) return s;
		std::cerr << "internal error: unknown flag " << flag << std::endl;
		ExitNow(1);
	}
	static std::string ArgId(const ArgSpec& s) { return std::string("Argument: -") + s.flag + " (--" + s.name + ")"; }

	void Usage(std::ostream& out, bool full) const
	{
		out << (full ? "USAGE: " : "Brief USAGE: ") << std::endl << "   " << mProg;
		for (auto& s : mSpecs)
		{
			out << " ";
			if (!s.required) out << "[";
			out << "-" << s.flag << " <" << s.type_desc << ">";
			if (!s.required) out << "]";
		}
		out << " [--] [--version] [-h]" << std::endl;
		if (full)
		{
			out << std::endl << "Where: " << std::endl;
			for (auto& s : mSpecs)
				out << "   -" << s.flag << " <" << s.type_desc << ">,  --" << s.name << " <" << s.type_desc << ">" << std::endl
				    << "     " << (s.required ? "(required)  " : "") << s.desc << std::endl << std::endl;
			out << "   " << mDesc << std::endl;
		}
	}

	[[noreturn]] void Fail(const std::string& arg_id, const std::string& what) const
	{
		std::cerr << "PARSE ERROR: " << arg_id << std::endl << "             " << what << std::endl << std::endl;
		Usage(std::cerr, false);
		std::cerr << std::endl << "For complete USAGE and HELP type: " << std::endl << "   " << mProg << " --help" << std::endl << std::endl;
		ExitNow(1);
	}

	std::string mProg;
	std::string mDesc;
	std::vector<ArgSpec> mSpecs;
};

// ---------------------------------------------------------------------------------------------
// small parsing helpers with the strictness the reference gets from boost
// ---------------------------------------------------------------------------------------------

// split on a single character, empty tokens kept (boost::split + is_any_of, no token compression)
inline void SplitChar(const std::string& s, char sep, std::vector<std::string>& out)
{
	out.clear();
	size_t start = 0;
	for (;;)
	{
		size_t p = s.find(sep, start);
		if (p == std::string::npos)
		{
			out.emplace_back(s, start);
			return;
		}
		out.emplace_back(s, start, p - start);
		start = p + 1;
	}
}

// lexical_cast<int>: the whole token must be one decimal integer (optional sign), else false
inline bool ParseInt(const std::string& s, int& out)
{
	if (s.empty()) return false;
	size_t i = 0;
	bool neg = false;
	if (s[0] == '-' || s[0] == '+')
	{
		neg = s[0] == '-';
		i = 1;
	}
	if (i >= s.size()) return false;
	long long v = 0;
	for (; i < s.size(); i++)
	{
		if (s[i] < '0' || s[i] > '9') return false;
		v = v * 10 + (s[i] - '0');
		if (v > 4294967296LL) return false;
	}
	if (neg) v = -v;
	if (v < -2147483648LL || v > 2147483647LL) return false;
	out = (int)v;
	return true;
}

// the reference lets a bad_lexical_cast escape from most call sites: terminate -> abort.  We report and exit 1.
inline int IntOrDie(const std::string& s, const char* what)
{
	int v = 0;
	if (!ParseInt(s, v))
	{
		std::cerr << "Error: bad lexical cast: " << what << " '" << s << "'" << std::endl;
		ExitNow(1);
	}
	return v;
}

// reverse, then complement ACGTacgt only; every other byte is kept (tools/Common.cpp:32-54)
inline void ReverseComplementInPlace(std::string& s)
{
	static unsigned char table[256];
	static bool init = false;
	if (!init)
	{
		for (int k = 0; k < 256; k++) table[k] = (unsigned char)k;
		const char* from = "ACGTacgt";
		const char* to = "TGCAtgca";
		for (int k = 0; k < 8; k++) table[(unsigned char)from[k]] = (unsigned char)to[k];
		init = true;
	}
	const size_t n = s.size();
	for (size_t lo = 0, hi = n; lo < hi;)
	{
		hi--;
		if (lo == hi)
		{
			s[lo] = (char)table[(unsigned char)s[lo]];
			break;
		}
		const unsigned char a = table[(unsigned char)s[lo]], b = table[(unsigned char)s[hi]];
		s[lo] = (char)b;
		s[hi] = (char)a;
		lo++;
	}
}

// union views of tools/Common.h:192-218: {index:31, end:1} as one int (hash key, output field)
inline int PackId(int index, int end) { return (int)(((unsigned)index & 0x7fffffffu) | ((unsigned)end << 31)); }
inline int IdIndex(int id) { return (int)((unsigned)id & 0x7fffffffu); }
inline int IdEnd(int id) { return (int)((unsigned)id >> 31); }

// ---------------------------------------------------------------------------------------------
// FASTQ: four lines per read, "@<fragment>/<1|2>" (tools/ReadStream.cpp:59-103)
// ---------------------------------------------------------------------------------------------
struct FastqRead
{
	std::string fragment;
	int read_end;
	std::string sequence;
};

class FastqReader
{
public:
	// nullptr semantics of IReadStream::Create (tools/ReadStream.cpp:21-51): extension must be fastq/fq, file must open
	bool Open(const std::string& filename)
	{
		const std::string::size_type dot = filename.find_last_of('.');
		const std::string ext = filename.substr(dot + 1);
		if (ext != "fastq" && ext != "fq")
		{
			std::cerr << "Error: unrecognized extension " << ext << std::endl;
			return false;
		}
		mFile = fopen(filename.c_str(), "rb");
		if (!mFile)
		{
			std::cerr << "Error: unable to open file " << filename << std::endl;
			return false;
		}
		setvbuf(mFile, nullptr, _IOFBF, 1 << 22);
		return true;
	}
	~FastqReader()
	{
		if (mFile) fclose(mFile);
	}
	bool Next(FastqRead& read)
	{
		std::string line[4];
		for (int k = 0; k < 4; k++)
			if (!GetLine(line[k])) return false;
		if (line[0].empty() || line[0][0] != '@')
		{
			std::cerr << "Error: Unable to interpret read name " << line[0] << std::endl;
			return false;
		}
		const std::string::size_type slash = line[0].find_first_of('/');
		// (the reference's guard here can never fire: `npos && ...`; a name without '/' falls through to the
		// read-end test below, exactly as it does there)
		const char end_name = (slash == std::string::npos || slash + 1 >= line[0].size()) ? '\0' : line[0][slash + 1];
		if (end_name != '1' && end_name != '2')
		{
			std::cerr << "Error: Unable to interpret read end " << line[0] << std::endl;
			return false;
		}
		read.fragment = line[0].substr(1, slash - 1);
		read.read_end = end_name == '1' ? 0 : 1;
		read.sequence.swap(line[1]);
		return true;
	}

private:
	bool GetLine(std::string& out)
	{
		out.clear();
		if (!mFile) return false;
		char* buf = nullptr;
		size_t cap = 0;
		(void)cap;
		(void)buf;
		int c;
		bool any = false;
		while ((c = getc_unlocked(mFile)) != EOF)
		{
			any = true;
			if (c == '\n') return true;
			out.push_back((char)c);
		}
		return any; // last line without newline still counts, like std::getline
	}
	FILE* mFile = nullptr;
};

// ---------------------------------------------------------------------------------------------
// GPU context shared by a tool
// ---------------------------------------------------------------------------------------------
// A context on one GPU.  CUDA start-up costs 2-3 s on a B200 box, so the context is created on a helper thread
// the moment the tool starts and only joined at the first use: parsing the inputs runs underneath it.
// The one device of a single-GPU tool run (DFB_DEVICE, default 0).  Nothing has touched CUDA yet: show the runtime only
// that device.  On a multi-GPU host the first CUDA call otherwise initialises every GPU of the box, which is most of a
// short tool run's wall time.
inline int SingleDevice()
{
	int dev = getenv("DFB_DEVICE") ? atoi(getenv("DFB_DEVICE")) : 0;
	if (dev >= 0 && !getenv("CUDA_VISIBLE_DEVICES"))
	{
		setenv("CUDA_VISIBLE_DEVICES", std::to_string(dev).c_str(), 1);
		dev = 0;
	}
	return dev;
}

class Gpu
{
public:
	Gpu() : Gpu(SingleDevice()) {}
	explicit Gpu(int device) : mDevice(device)
	{
		mThread = std::thread([this] {
			mStatus = dfb_ctx_create(mDevice, &mCtx);
			if (mStatus != DFB_OK) mError = dfb_last_error(nullptr);
		});
	}
	~Gpu()
	{
		if (mThread.joinable()) mThread.join();
		dfb_ctx_destroy(mCtx);
	}
	dfb_ctx* ctx()
	{
		if (mThread.joinable()) mThread.join();
		if (mStatus != DFB_OK)
		{
			std::cerr << "Error: " << mError << std::endl;
			ExitNow(1);
		}
		return mCtx;
	}
	[[noreturn]] void Die(const char* what)
	{
		std::cerr << "Error: " << what << ": " << dfb_last_error(mCtx) << std::endl;
		ExitNow(1);
	}
	Gpu(const Gpu&) = delete;
	Gpu& operator=(const Gpu&) = delete;

private:
	int mDevice;
	dfb_ctx* mCtx = nullptr;
	int mStatus = DFB_OK;
	std::string mError;
	std::thread mThread;
};

// The tools end like the reference's do (return from main), minus the seconds CUDA spends tearing its context
// down: outputs are flushed, then the process leaves without running the teardown.
[[noreturn]] inline void FinishProcess(int code)
{
	std::cout.flush();
	std::cerr.flush();
	fflush(nullptr);
	_exit(code);
}

// Devices a tool may use: DFB_DEVICES="0,1,2" or "all" (every visible GPU); else the single DFB_DEVICE (default 0).
inline std::vector<int> DeviceList()
{
	std::vector<int> out;
	const char* e = getenv("DFB_DEVICES");
	if (e && *e)
	{
		if (std::string(e) == "all")
		{
			const int n = dfb_device_count();
			for (int k = 0; k < n; k++) out.push_back(k);
		}
		else
		{
			std::vector<std::string> f;
			SplitChar(e, ',', f);
			for (const std::string& t : f)
			{
				int v = 0;
				if (ParseInt(t, v)) out.push_back(v);
			}
		}
	}
	if (out.empty()) out.push_back(SingleDevice());
	return out;
}

// DFB_TRACE=1: phase timings of a tool on stderr (stdout / the -a file stay byte-exact); `label` goes in front of
// every line (dosplitalign_multi: which split)
class PhaseTimer
{
public:
	explicit PhaseTimer(std::string label = "")
	    : mOn(getenv("DFB_TRACE") && *getenv("DFB_TRACE") && *getenv("DFB_TRACE") != '0'), mLabel(std::move(label))
	{
		clock_gettime(CLOCK_MONOTONIC, &mT);
	}
	void Lap(const char* what)
	{
		if (!mOn) return;
		timespec t;
		clock_gettime(CLOCK_MONOTONIC, &t);
		fprintf(stderr, "[tool] %s%-28s %9.3f ms\n", mLabel.c_str(), what, (t.tv_sec - mT.tv_sec) * 1e3 + (t.tv_nsec - mT.tv_nsec) * 1e-6);
		mT = t;
	}
	// the next lap starts now (time spent waiting elsewhere is charged to no phase)
	void Restart() { clock_gettime(CLOCK_MONOTONIC, &mT); }

	// accumulating form for phases that repeat per batch: Add("name") charges the time since the last call to a
	// named bucket, Report() prints the buckets
	void Add(const char* what)
	{
		if (!mOn) return;
		timespec t;
		clock_gettime(CLOCK_MONOTONIC, &t);
		const double ms = (t.tv_sec - mT.tv_sec) * 1e3 + (t.tv_nsec - mT.tv_nsec) * 1e-6;
		mT = t;
		for (auto& b : mBuckets)
			if (b.first == what)
			{
				b.second += ms;
				return;
			}
		mBuckets.emplace_back(what, ms);
	}
	void Report()
	{
		for (auto& b : mBuckets) fprintf(stderr, "[tool] %s%-28s %9.3f ms\n", mLabel.c_str(), b.first.c_str(), b.second);
		mBuckets.clear();
	}

private:
	bool mOn;
	std::string mLabel;
	timespec mT;
	std::vector<std::pair<std::string, double>> mBuckets;
};

// CSR table under construction
struct TableBuilder
{
	std::string bytes;
	std::vector<int64_t> off{0};
	int64_t Add(const char* p, size_t n)
	{
		bytes.append(p, n);
		off.push_back((int64_t)bytes.size());
		return (int64_t)off.size() - 2;
	}
	int64_t Add(const std::string& s) { return Add(s.data(), s.size()); }
	int64_t Count() const { return (int64_t)off.size() - 1; }
	void Clear()
	{
		bytes.clear();
		off.assign(1, 0);
	}
	dfb_seq_table View() const { return dfb_seq_table{(const uint8_t*)bytes.data(), off.data(), Count()}; }
};

}  // namespace dfbhost
