// abawaca (B200): same command line, same inputs and same output files as the reference program
// (/root/reference/src/abawaca.cpp main, :54-217), with the whole recursive split search on the device:
//   the work list :98-197 + ClusterSeparatorBySensitivitySpecificity::separate()  ->  abw_search_create + abw_search_run
// The loaders below rebuild what ScafDpData (ScafDpData.cpp:11-120), ClusterData (ClusterData.cpp:27-168) and SCGdb
// (SCGdb.cpp:58-120) build, as flat arrays; the writers reproduce log, summary.txt, dp2cluster.txt, scaf2cluster.txt,
// final-clusters/<id>.fasta and clusters/<id>.{lrn,scaf-cluster.txt,scaf-stats.txt} from the records the device returns; the data lines of
// clusters/<id>.lrn (abw_format_lrn) and the text of final-clusters/<id>.fasta (abw_fasta_format / abw_twobit_format) are made on the device, where the
// assembly stays from loading to the last bin.
#include "abw_host.h"
#include <algorithm>
#include <cmath>
#include <ctime>
#include <fstream>
#include <iostream>
#include <set>

using namespace abwh;

#define VERSION "v1.07"

static const char* get_time()
{
	static time_t t0 = time(nullptr);
	static char str[64];
	int t = (int)(time(nullptr) - t0);
	snprintf(str, sizeof(str), "%02i:%02i:%02i", t / 3600, (t % 3600) / 60, t % 60);
	return str;
}

struct Params {
	std::string lrn_file, names_file, info_file, links_file, fasta_file, root_dir, gene2scg_file;
	std::string scg_list_file = "/home/itaish/software/cpp/abawaca/curr-version/scg.list";   // abawaca.cpp:42; $ABW_SCG_LIST overrides it here
	std::string build_dir, cluster_dir, fasta_dir;
	bool scg_from_cli = false;          // -c was given: it wins over the SCG line of data.txt whatever the order of the flags
	int ncpus = 1;          // accepted and checked like the reference (1..40); the device does not need it
	int strategy = ABW_SENS_SPEC;
};

static void usage(const char* prog)
{
	fprintf(stderr, "Usage: %s -u <abawaca-build-directory> -f <fasta-file> -o <out-dir> [-p <# CPUs>] [-c <gene2scg>]\n\n", prog);
}

static int read_params(Params& P, int argc, const char** argv)
{
	if(argc == 1 || (argc == 2 && (!strcmp(argv[1], "-h") || !strcmp(argv[1], "--help")))) {
		usage(argv[0]);
		return -1;
	}
	for(int i = 1; i < argc; i++) {
		if(!strcmp(argv[i], "-u") && i + 1 < argc) {
			P.build_dir = argv[++i];
			const std::string data_file = P.build_dir + "/data.txt";
			FILE* fp = fopen(data_file.c_str(), "r");
			if(!fp) {
				std::cerr << "Error: could not find " << P.build_dir << "/data.txt. Is it possible that the data was generated using an old version of abawaca-build? (prior to v1.07)"
				          << std::endl << std::endl;
				return -1;
			}
			char line[8192];
			while(fgets(line, sizeof(line), fp)) {
				size_t n = strlen(line);
				while(n > 0 && line[n - 1] == '\n') line[--n] = 0;
				char* p = strchr(line, '\t');
				if(!p) continue;
				*(p++) = 0;
				while(*p && isspace((unsigned char)*p)) p++;
				if(!strcmp(line, "Links")) P.links_file = p;
				else if(!strcmp(line, "Info")) P.info_file = p;
				else if(!strcmp(line, "Names")) P.names_file = p;
				else if(!strcmp(line, "Lrn")) P.lrn_file = p;
				else if(!strcmp(line, "Assembly")) P.fasta_file = p;
				else if(!strcmp(line, "SCG")) { if(!P.scg_from_cli) P.gene2scg_file = p; }
			}
			fclose(fp);
		}
		else if(!strcmp(argv[i], "-f") && i + 1 < argc) P.fasta_file = argv[++i];
		else if(!strcmp(argv[i], "-o") && i + 1 < argc) P.root_dir = argv[++i];
		else if(!strcmp(argv[i], "-p") && i + 1 < argc) {
			P.ncpus = atoi(argv[++i]);
			if(P.ncpus == 0 || P.ncpus > 40) {
				std::cerr << "Error: # CPUs (" << argv[i] << ") must be an integer between 1 to 40" << std::endl << std::endl;
				return -1;
			}
		}
		else if(!strcmp(argv[i], "-c") && i + 1 < argc) { P.gene2scg_file = argv[++i]; P.scg_from_cli = true; }
		else if(!strcmp(argv[i], "--split-scafs")) P.strategy = ABW_SPLIT_SCAFS;   // the alternative strategy the reference compiles but never selects (abawaca.cpp:110)
		else {
			std::cerr << "Unrecognizes flag: " << argv[i] << std::endl;
			return -1;
		}
	}
	if(const char* e = getenv("ABW_SCG_LIST"))
		P.scg_list_file = e;
	if(P.lrn_file.empty()) {
		std::cerr << "abawaca-build directrory was not specified (-u)" << std::endl << std::endl;
		return -1;
	}
	struct { const std::string* f; const char* what; } need[] = {{&P.names_file, "names"}, {&P.lrn_file, "lrn"}, {&P.info_file, "info"}, {&P.links_file, "links"}};
	for(auto& nf : need)
		if(!file_readable(*nf.f)) {
			std::cerr << "Could not read " << nf.what << " file (" << *nf.f << ") from the abawaca directory (" << P.build_dir << ")" << std::endl;
			return -1;
		}
	if(!file_readable(P.fasta_file)) { std::cerr << "Could not read " << P.fasta_file << std::endl; return -1; }
	if(!P.gene2scg_file.empty() && !file_readable(P.gene2scg_file)) {
		if(P.scg_from_cli) { std::cerr << "Could not read " << P.gene2scg_file << std::endl; return -1; }
		// the path came from data.txt and abawaca-build could not produce the file (no gene caller on this host): run without an SCG database
		std::cerr << "Warning: " << P.gene2scg_file << " (SCG line of data.txt) is not readable; continuing without SCG information (pass -c <gene2scg>)" << std::endl;
		P.gene2scg_file.clear();
	}
	if(!file_readable(P.scg_list_file)) { std::cerr << "Could not read " << P.scg_list_file << std::endl; return -1; }
	P.cluster_dir = P.root_dir + "/clusters";
	P.fasta_dir = P.root_dir + "/final-clusters";
	for(const std::string* d : {&P.root_dir, &P.cluster_dir, &P.fasta_dir})
		if(!directory_exists(*d)) {
			std::string cmd = "mkdir " + *d;
			if(system(cmd.c_str()) != 0)
				std::cerr << "Warning: could not create " << *d << std::endl;
		}
	return 0;
}

// ---- the data model as flat arrays ------------------------------------------------------------------------------------------------
struct Model {
	// scaffolds (1-based ids = index + 1, name order) and datapoints (1-based ids, (scaffold, dp name) order)
	std::vector<std::string> scaf_names;
	std::vector<uint32_t> scaf_rec;             // record of the scaffold in the assembly file
	std::vector<double> scaf_cvg, scaf_gc;
	std::vector<uint32_t> T;
	std::vector<uint64_t> len;
	std::vector<uint32_t> dp2scaf;              // 0-based scaffold of 0-based dp
	std::vector<unsigned long> dp_name;
	std::vector<std::string> dim_names;
	std::vector<double> rows;                   // the .lrn rows in file order, row major [rows][D]
	std::vector<uint64_t> row_of_dp;            // row of rows of 0-based dp
	double* d_rows = nullptr;                   // on the device in dp order, row major [N][D]: what the search reads and the cluster dumps print
	std::vector<uint64_t> scgmask;              // [S][W]
	uint32_t W = 1;
	int total_num_scgs = 0;
	// the assembly on the device: FASTA text indexed by abw_fasta_scan, or a .2bit image (d_file) parsed by abw_twobit_scan
	abw_fasta* fa = nullptr;
	abw_twobit* tb = nullptr;
	void* d_file = nullptr;
	size_t N() const { return dp2scaf.size(); }
	size_t S() const { return scaf_names.size(); }
	size_t D() const { return dim_names.size(); }
};

static void load_model(const Params& P, Model& M, abw_ctx* ctx)
{
	// .info: scaffold -> coverage (ScafDpData.cpp:21-32)
	std::map<std::string, double> name2cvg;
	{
		FILE* fp = fopen(P.info_file.c_str(), "r");
		if(!fp) throw std::invalid_argument("could not read " + P.info_file);
		char line[8192], name[512];
		while(fgets(line, sizeof(line), fp)) {
			unsigned long length, Ns;
			double cvg, gc;
			if(sscanf(line, "%511s %lu %lf %lf %lu", name, &length, &cvg, &gc, &Ns) != 5) {
				fclose(fp);
				throw std::invalid_argument("Illegal line in file " + P.info_file + ":\n" + line);
			}
			name2cvg.insert(std::make_pair(std::string(name), cvg));
		}
		fclose(fp);
	}
	// .names (ScafDpData.cpp:41-87): dp name, window name, "<scaf>:(<s>, <e>), <nonN>/<len> non-Ns bps"
	std::map<std::string, std::set<unsigned long>> scaf2dps;
	{
		FILE* fp = fopen(P.names_file.c_str(), "r");
		if(!fp) throw std::invalid_argument("could not read " + P.names_file);
		char line[8192];
		if(!fgets(line, sizeof(line), fp)) { fclose(fp); throw std::invalid_argument("file " + P.names_file + " is empty"); }
		unsigned t1; char c;
		if(sscanf(line, "%c %u", &c, &t1) != 2 || c != '%') { fclose(fp); throw std::invalid_argument("unexpected line in file " + P.names_file + ":\n" + line); }
		while(fgets(line, sizeof(line), fp)) {
			char* marks[5] = {strchr(line, ':'), strchr(line, '('), strchr(line, ')'), strchr(line, '/'), strchr(line, ',')};
			for(char* m : marks)
				if(!m) { fclose(fp); throw std::invalid_argument("unexpected line in file " + P.names_file + ":\n" + line); }
			for(char* m : marks) *m = ' ';
			unsigned long dp = 0, start = 0, end = 0, a = 0, b = 0, cc = 0;
			char seg[512], scaf[512];
			if(sscanf(line, "%lu %511s %511s %lu %lu , %lu segment(s), %lu %lu non-N bps", &dp, seg, scaf, &start, &end, &cc, &a, &b) != 8 &&
			   sscanf(line, "%lu %511s %511s %lu %lu , %lu %lu non-N bps", &dp, seg, scaf, &start, &end, &a, &b) != 7) {
				fclose(fp);
				throw std::invalid_argument("unexpected line in file " + P.names_file + ":\n" + line);
			}
			scaf2dps[scaf].insert(dp);
		}
		fclose(fp);
	}
	std::map<unsigned long, size_t> dp_name2id;    // 1-based internal id
	std::map<std::string, size_t> scaf_name2id;
	for(auto& kv : scaf2dps) {
		if(kv.second.size() == 1)
			continue;                                // ScafDpData.cpp:92-93
		scaf_name2id[kv.first] = M.scaf_names.size() + 1;
		M.scaf_names.push_back(kv.first);
		M.T.push_back((uint32_t)kv.second.size());
		for(unsigned long dpn : kv.second) {
			M.dp2scaf.push_back((uint32_t)(M.scaf_names.size() - 1));
			M.dp_name.push_back(dpn);
			dp_name2id[dpn] = M.dp2scaf.size();
		}
	}
	// assembly: read once, kept on the device for the bin files
	{
		std::string bytes = read_file(P.fasta_file);
		const bool twobit = is_twobit(bytes);
		if(twobit? abw_twobit_scan(ctx, bytes.data(), bytes.size(), &M.tb) != ABW_OK : abw_fasta_scan(ctx, bytes.data(), bytes.size(), 0, &M.fa) != ABW_OK)
			throw std::runtime_error(std::string(abw_last_error(ctx)) + " (" + P.fasta_file + ")");
		if(twobit) {
			ABWH_CHECK(ctx, abw_device_alloc(ctx, std::max<size_t>(bytes.size(), 1), &M.d_file));
			ABWH_CHECK(ctx, abw_copy_to_device(ctx, M.d_file, bytes.data(), bytes.size()));
		}
		const uint64_t nrec = twobit? abw_twobit_count(M.tb) : abw_fasta_count(M.fa);
		std::vector<uint64_t> id_off(nrec), rec_len(nrec), count_N(nrec), count_GC(nrec);
		std::vector<uint32_t> id_len(nrec);
		if(twobit) {
			ABWH_CHECK(ctx, abw_twobit_get(ctx, M.tb, id_off.data(), id_len.data(), rec_len.data()));
			ABWH_CHECK(ctx, abw_twobit_base_counts(ctx, M.tb, M.d_file, 0, count_N.data(), count_GC.data()));
		}
		else {
			ABWH_CHECK(ctx, abw_fasta_get(ctx, M.fa, id_off.data(), id_len.data(), rec_len.data()));
			ABWH_CHECK(ctx, abw_fasta_base_counts(ctx, M.fa, count_N.data(), count_GC.data()));
		}
		const uint32_t none = 0xFFFFFFFFu;
		M.scaf_rec.assign(M.S(), none);
		M.scaf_cvg.assign(M.S(), 0);
		for(uint64_t i = 0; i < nrec; i++) {
			const std::string id = bytes.substr(id_off[i], id_len[i]);
			auto it = scaf_name2id.find(id);
			if(it != scaf_name2id.end()) {                 // a repeated id overwrites the earlier record (scafs[id] = Seq(...), ScafDpData.cpp:110)
				M.scaf_rec[it->second - 1] = (uint32_t)i;
				auto ci = name2cvg.find(id);
				M.scaf_cvg[it->second - 1] = (ci == name2cvg.end())? 0 : ci->second;
			}
		}
		M.len.resize(M.S());
		M.scaf_gc.resize(M.S());
		for(size_t s = 0; s < M.S(); s++) {
			const uint32_t r = M.scaf_rec[s];
			if(r == none)
				throw std::invalid_argument("scaffold " + M.scaf_names[s] + " is not in " + P.fasta_file);
			M.len[s] = rec_len[r];
			// Bio::gc after DNAString upper-casing (String.cpp:114-131)
			M.scaf_gc[s] = (rec_len[r] == count_N[r])? 0 : (double)count_GC[r] / (double)(rec_len[r] - count_N[r]);
		}
	}
	// .lrn (ClusterData.cpp:27-168)
	{
		FILE* fp = fopen(P.lrn_file.c_str(), "r");
		if(!fp) { std::cerr << "Fatal error: could not read " << P.lrn_file << std::endl << std::endl; exit(-1); }
		char* line = nullptr; size_t cap = 0; ssize_t n;
		unsigned ndps = 0, ndims = 0; char c;
		auto next = [&]() { n = getline(&line, &cap, fp); return n >= 0; };
		if(!next() || sscanf(line, "%c %u", &c, &ndps) != 2 || c != '%') { std::cerr << "Fatal error: unexpected line 1 in " << P.lrn_file << std::endl; exit(-1); }
		if(!next() || sscanf(line, "%c %u", &c, &ndims) != 2 || c != '%') { std::cerr << "Fatal error: unexpected line 2 in " << P.lrn_file << std::endl; exit(-1); }
		ndims--;
		if(!next()) { std::cerr << "Fatal error: failed to read line 3 in " << P.lrn_file << std::endl; exit(-1); }
		{
			unsigned t = 1;
			for(char* p = line; *p; p++) t += (*p == '\t');
			if(t != ndims + 1) { std::cerr << "Fatal error: unexpected line 3 in " << P.lrn_file << std::endl; exit(-1); }
		}
		if(!next()) { std::cerr << "Fatal error: failed to read line 4 in " << P.lrn_file << std::endl; exit(-1); }
		while(n > 0 && isspace((unsigned char)line[n - 1])) line[--n] = 0;
		{
			char* p = strchr(line, '\t');
			while(p) {
				char* q = strchr(p + 1, '\t');
				M.dim_names.push_back(q? std::string(p + 1, q) : std::string(p + 1));
				p = q;
			}
			if(M.dim_names.size() != ndims) { std::cerr << "Fatal error: number of dimensions found in line 4 (" << M.dim_names.size() << ") is different than expected (" << ndims << ")" << std::endl; exit(-1); }
		}
		const size_t N = M.N(), D = ndims;
		std::vector<char> seen(N, 0);
		// the datapoint lines are parsed on the device (abw_parse_lrn): keys and a row-major matrix come back
		std::string body;
		{
			char buf[1 << 16];
			size_t got;
			while((got = fread(buf, 1, sizeof(buf), fp)) > 0)
				body.append(buf, got);
		}
		free(line);
		fclose(fp);
		uint64_t cap_rows = 1;
		for(char ch : body) cap_rows += (ch == '\n');
		uint64_t* d_keys = nullptr;
		double* d_vals = nullptr;
		ABWH_CHECK(ctx, abw_device_alloc(ctx, cap_rows * sizeof(uint64_t), (void**)&d_keys));
		ABWH_CHECK(ctx, abw_device_alloc(ctx, std::max<uint64_t>(cap_rows * D, 1) * sizeof(double), (void**)&d_vals));
		uint64_t entry = 0;
		if(abw_parse_lrn(ctx, body.data(), body.size(), 0, (uint32_t)D, d_keys, d_vals, cap_rows, &entry) != ABW_OK) {
			std::cerr << "Fatal error: " << abw_last_error(ctx) << ", file " << P.lrn_file << std::endl;
			exit(-1);
		}
		if(entry > ndps) { std::cerr << "Fatal error: number of datapoint lines found is higher than expected (" << ndps << "), file " << P.lrn_file << std::endl; exit(-1); }
		if(entry != ndps) { std::cerr << "Fatal error: number of datapoint lines found (" << entry << ") is different than expected (" << ndps << "), file " << P.lrn_file << std::endl; exit(-1); }
		std::vector<uint64_t> keys(entry);
		M.rows.resize(entry * D);
		if(entry) {
			ABWH_CHECK(ctx, abw_copy_to_host(ctx, keys.data(), d_keys, entry * sizeof(uint64_t)));
			ABWH_CHECK(ctx, abw_copy_to_host(ctx, M.rows.data(), d_vals, entry * D * sizeof(double)));
		}
		ABWH_CHECK(ctx, abw_device_free(ctx, d_keys));
		M.row_of_dp.assign(N, 0);
		for(uint64_t r = 0; r < entry; r++) {
			auto it = dp_name2id.find((unsigned long)keys[r]);
			if(it != dp_name2id.end()) {
				const size_t dp = it->second - 1;
				seen[dp] = 1;
				M.row_of_dp[dp] = r;
			}
		}
		for(size_t i = 0; i < N; i++)
			if(!seen[i])
				throw std::invalid_argument("datapoint " + std::to_string(M.dp_name[i]) + " of " + P.names_file + " has no row in " + P.lrn_file);
		// the rows of the file put into dp order where they already are, for the search and the cluster dumps
		ABWH_CHECK(ctx, abw_device_alloc(ctx, std::max<size_t>(N * D, 1) * sizeof(double), (void**)&M.d_rows));
		ABWH_CHECK(ctx, abw_gather_rows(ctx, d_vals, D, M.row_of_dp.data(), 0, N, (uint32_t)D, M.d_rows, D));
		ABWH_CHECK(ctx, abw_device_free(ctx, d_vals));
	}
	// SCG database (SCGdb.cpp:58-120): number of names in scg.list; gene -> SCG, gene = <scaffold>_<non-zero integer>
	{
		FILE* fp = fopen(P.scg_list_file.c_str(), "r");
		if(!fp) throw std::invalid_argument("Failed to read file " + P.scg_list_file);
		char tok[1024];
		while(fscanf(fp, "%1023s", tok) == 1) M.total_num_scgs++;
		fclose(fp);
		std::map<std::string, uint32_t> scg_index;
		std::vector<std::pair<uint32_t, uint32_t>> hits;
		if(!P.gene2scg_file.empty()) {
			fp = fopen(P.gene2scg_file.c_str(), "r");
			if(!fp) throw std::invalid_argument("Failed to read file " + P.gene2scg_file);
			char gene[1024], scg[1024];
			while(fscanf(fp, "%1023s %1023s", gene, scg) == 2) {
				char* p = strrchr(gene, '_');
				if(!p) { fclose(fp); throw std::invalid_argument(std::string("Unexpected gene name ") + gene + ", expected prodigal format: <name>_<integer>"); }
				*p = 0;
				auto it = scaf_name2id.find(gene);
				if(it == scaf_name2id.end())
					continue;
				if(atoi(p + 1) == 0) { fclose(fp); throw std::invalid_argument(std::string("Could not identify gene id in ") + gene + "_" + (p + 1)); }
				auto si = scg_index.insert(std::make_pair(std::string(scg), (uint32_t)scg_index.size())).first;
				hits.push_back(std::make_pair((uint32_t)(it->second - 1), si->second));
			}
			fclose(fp);
		}
		M.W = std::max<uint32_t>(1, (uint32_t)((scg_index.size() + 63) / 64));
		M.scgmask.assign(M.S() * M.W, 0);
		for(auto& h : hits)
			M.scgmask[(size_t)h.first * M.W + h.second / 64] |= 1ull << (h.second % 64);
	}
}

// The FASTA text of the assembly records `recs` (abw_fasta_format / abw_twobit_format) in windows of LRN_CHUNK bytes: d_text (LRN_CHUNK bytes of device
// memory) and text are scratch, kept from file to file.  false when fp takes fewer bytes than it is given.
static bool write_fasta(abw_ctx* ctx, FILE* fp, const Model& M, const std::vector<uint32_t>& recs, char* d_text, std::vector<char>& text)
{
	for(uint64_t byte0 = 0, total = 1; byte0 < total;) {
		uint64_t nbytes = 0;
		if(M.tb)
			ABWH_CHECK(ctx, abw_twobit_format(ctx, M.tb, M.d_file, 0, recs.data(), recs.size(), byte0, d_text, LRN_CHUNK, &total, &nbytes));
		else
			ABWH_CHECK(ctx, abw_fasta_format(ctx, M.fa, recs.data(), recs.size(), byte0, d_text, LRN_CHUNK, &total, &nbytes));
		text.resize(std::max<size_t>(text.size(), nbytes));
		if(nbytes)
			ABWH_CHECK(ctx, abw_copy_to_host(ctx, text.data(), d_text, nbytes));
		if(fwrite(text.data(), 1, nbytes, fp) != nbytes)
			return false;
		byte0 += nbytes;
	}
	return true;
}

// size-weighted mean and standard deviation in scaffold-id order (ClusterQuality.cpp:6-27)
static void weighted_stats(const std::vector<std::pair<size_t, double>>& data, double& mean, double& stdev)
{
	if(data.empty()) { mean = stdev = -1; return; }
	size_t total = 0;
	mean = 0; stdev = 0;
	for(auto& d : data) { mean += d.first * d.second; total += d.first; }
	mean /= total;
	for(auto& d : data) stdev += d.first * (d.second - mean) * (d.second - mean);
	stdev = sqrt(stdev / (total - 1));
}

int main(int argc, const char** argv)
{
	milestone("start");
	std::cerr << "abawaca " << VERSION << std::endl << std::endl;
	Params P;
	if(read_params(P, argc, argv))
		return -1;
	std::ofstream log((P.root_dir + "/log").c_str()), summary((P.root_dir + "/summary.txt").c_str()), ofs_dp((P.root_dir + "/dp2cluster.txt").c_str()),
	              ofs_scaf((P.root_dir + "/scaf2cluster.txt").c_str());
	std::cerr << '[' << get_time() << ']' << " Starting" << std::endl;
	std::cerr << '[' << get_time() << ']' << " Creating databases based on " << P.names_file << " and " << P.lrn_file << std::endl;
	log << "abawaca " << VERSION << std::endl << std::endl;
	log << '[' << get_time() << ']' << " Starting" << std::endl;
	log << '[' << get_time() << ']' << " Creatinf databases based on " << P.names_file << " and " << P.lrn_file << std::endl;
	try {
		abw_ctx* ctx = nullptr;
		if(abw_ctx_create(0, &ctx) != ABW_OK) {
			std::cerr << "Error: no usable CUDA device (abawaca_b200 has no CPU path)" << std::endl;
			return -1;
		}
		milestone("abw_ctx_create");
		Model M;
		load_model(P, M, ctx);
		milestone("load_model");
		const size_t N = M.N(), S = M.S(), D = M.D();
		summary << "Cluster\t# scafs\t# dps\t# bps\t%G+C\tStdev\tCvg\tstdev\t#SCG" << '/' << M.total_num_scgs << "\tAvg" << std::endl;

		abw_params prm;
		abw_default_params(&prm);
		prm.min_reported_score = 0;                 // also report the best separation of terminal clusters, as the reference's log does
		abw_search* search = nullptr;
		// the search reads M.d_rows where it lies: it is freed after abw_search_destroy
		ABWH_CHECK(ctx, abw_search_create(ctx, M.d_rows, 1, ABW_LAYOUT_ROWMAJOR, D, N, nullptr, N, (uint32_t)D, M.dp2scaf.data(), (uint32_t)S, M.T.data(), M.len.data(),
		                                  M.scgmask.data(), M.W, &prm, P.strategy, &search));
		std::vector<abw_cluster_rec> recs(2 * N / std::max<uint32_t>(prm.cluster_ndps_threshold, 1) + 64);
		std::vector<uint32_t> dp2cluster(N), scaf2cluster(S);
		uint32_t nrec = 0;
		ABWH_CHECK(ctx, abw_search_set_scaffold_stats(ctx, search, M.scaf_gc.data(), M.scaf_cvg.data()));
		ABWH_CHECK(ctx, abw_search_run(ctx, search, recs.data(), (uint32_t)recs.size(), &nrec, dp2cluster.data(), scaf2cluster.data()));
		if(nrec > recs.size()) {
			std::cerr << "Fatal error: " << nrec << " clusters were evaluated but only " << recs.size() << " records fit" << std::endl;
			return -1;
		}
		recs.resize(nrec);
		milestone("search");

		// membership of every evaluated cluster: terminal bins bubble up to their ancestors
		std::map<uint32_t, uint32_t> parent_of;
		for(auto& r : recs) parent_of[r.id] = r.parent;
		std::map<uint32_t, std::vector<uint32_t>> dps_of;      // 0-based datapoints, ascending
		for(size_t i = 0; i < N; i++)
			for(uint32_t c = dp2cluster[i]; c != 0; c = parent_of[c]) dps_of[c].push_back((uint32_t)i);
		// scratch of the cluster dumps (write_lrn) and the bin files (write_fasta)
		char* d_text = nullptr;
		ABWH_CHECK(ctx, abw_device_alloc(ctx, LRN_CHUNK, (void**)&d_text));
		std::vector<char> text;
		std::vector<uint64_t> rows;
		std::vector<uint32_t> recs_of_bin;
		auto gc_cvg_of = [&](const std::vector<uint32_t>& assigned, double& avg_gc, double& sd_gc, double& avg_cvg, double& sd_cvg) {
			std::vector<std::pair<size_t, double>> gc, cvg;
			for(uint32_t s : assigned) {
				gc.push_back(std::make_pair((size_t)M.len[s], M.scaf_gc[s]));
				cvg.push_back(std::make_pair((size_t)M.len[s], M.scaf_cvg[s]));
			}
			weighted_stats(gc, avg_gc, sd_gc);
			weighted_stats(cvg, avg_cvg, sd_cvg);
		};

		// assigned scaffolds per cluster: root = all; children = vote of the split (ClusterSeparator.cpp:94-101) on the winning dimension
		std::map<uint32_t, std::vector<uint32_t>> assigned_of;
		assigned_of[1].resize(S);
		for(size_t s = 0; s < S; s++) assigned_of[1][s] = (uint32_t)s;

		for(const abw_cluster_rec& r : recs) {
			const std::vector<uint32_t>& cur_dps = dps_of[r.id];
			std::cerr << std::endl << '[' << get_time() << ']' << " Checking cluster " << r.id << " (" << r.ndps << " datapoints)" << std::endl;
			log << std::endl << '[' << get_time() << ']' << " Checking cluster " << r.id << " (" << r.ndps << " datapoints)" << std::endl;
			auto print_params = [&](std::ostream& os) {
				if(r.best.found) os << "Dimension: " << (size_t)r.best.dim << ", value:" << r.best.value;
				else os << "Dimension: " << (size_t)-1 << ", value:" << -1.0;
				if(P.strategy == ABW_SENS_SPEC)
					os << ", Specificity: " << r.best.b << ", sensitivity:" << r.best.a;
			};
			std::cerr << '[' << get_time() << ']' << " "; print_params(std::cerr); std::cerr << std::endl;
			log << '[' << get_time() << ']' << " "; print_params(log); log << std::endl;
			if(!r.split) {
				std::cerr << '[' << get_time() << ']' << " Cluster " << r.id << " is a terminal cluster" << std::endl;
				log << '[' << get_time() << ']' << " Cluster " << r.id << " is a terminal cluster" << std::endl;
				const std::vector<uint32_t>& assigned = assigned_of[r.id];
				// final-clusters/<id>.fasta: 60 columns, one more (possibly empty) line when the length is a multiple of 60 (SeqIOWrite_fasta.h:40-51),
				// made on the device in windows of the dump scratch
				{
					const std::string path = P.fasta_dir + "/" + std::to_string(r.id) + ".fasta";
					FILE* fp = fopen(path.c_str(), "w");
					recs_of_bin.clear();
					for(uint32_t s : assigned) recs_of_bin.push_back(M.scaf_rec[s]);
					if(!fp || !write_fasta(ctx, fp, M, recs_of_bin, d_text, text)) {
						std::cerr << "Fatal error: could write to file " << path << std::endl << std::endl;
						exit(-1);
					}
					fclose(fp);
				}
				// ClusterQuality::scg, gc and cvg of the bin come back with its record (gc and cvg: abw_search_set_scaffold_stats)
				summary << r.id << '\t' << assigned.size() << '\t' << cur_dps.size() << '\t' << r.total_size << '\t' << int(1000 * r.gc_avg) / 10.0 << '\t' << int(1000 * r.gc_sd) / 100.0
				        << '\t' << int(10 * r.cvg_avg) / 10.0 << '\t' << int(10 * r.cvg_sd) / 10.0 << '\t' << r.scg_unique << '\t' << int(100 * r.scg_avg) / 100.0 << std::endl;
				continue;
			}
			// the split: raw sides on the winning dimension, then the vote (ClusterSeparator.cpp:25-54,82-134)
			std::vector<uint32_t> low, high;
			for(uint32_t dp : cur_dps) (M.rows[M.row_of_dp[dp] * D + r.best.dim - 1] <= r.best.value? low : high).push_back(dp);
			const bool swapped = high.size() < low.size();
			const std::vector<uint32_t>& raw1 = swapped? high : low;
			const std::vector<uint32_t>& raw2 = swapped? low : high;
			std::map<uint32_t, uint32_t> n1, n2;
			for(uint32_t dp : raw1) n1[M.dp2scaf[dp]]++;
			for(uint32_t dp : raw2) n2[M.dp2scaf[dp]]++;
			std::vector<uint32_t> a1, a2;
			for(auto& kv : n1) if(2ull * kv.second >= M.T[kv.first]) a1.push_back(kv.first);
			for(auto& kv : n2) if(2ull * kv.second > M.T[kv.first]) a2.push_back(kv.first);
			assigned_of[r.child1] = a1;
			assigned_of[r.child2] = a2;
			auto best_line = [&](std::ostream& os) {
				os << " Best separation:\t" << "dimension " << (size_t)r.best.dim << " (" << M.dim_names[r.best.dim - 1] << ")\t" << "Value " << r.best.value << "\t";
				if(P.strategy == ABW_SENS_SPEC) os << "Specificity " << r.best.b << "\t" << "Sensitivity " << r.best.a;
				else os << "best split scaf ratio " << r.best.a << std::endl;
			};
			std::cerr << '[' << get_time() << ']'; best_line(std::cerr); std::cerr << std::endl;
			std::cerr << '[' << get_time() << ']' << " Cluster " << r.id << " will be separated to the following two clusters" << std::endl;
			log << '[' << get_time() << ']'; best_line(log); log << std::endl;
			log << '[' << get_time() << ']' << " Cluster " << r.id << " will be separated to the following two clusters" << std::endl;
			const uint32_t child[2] = {r.child1, r.child2};
			const std::vector<uint32_t>* assigned[2] = {&a1, &a2};
			const std::vector<uint32_t>* raw[2] = {&raw1, &raw2};
			for(int ch = 0; ch < 2; ch++) {
				const std::vector<uint32_t>& cdps = dps_of[child[ch]];
				// <id>.lrn: "<dp+1>" and "\t%lf" per value (ClusterWriter.cpp:81-98); the reference writes the rows in unordered_set order (quirk Q9), here
				// ascending dp id
				{
					const std::string path = P.cluster_dir + "/" + std::to_string(child[ch]) + ".lrn";
					FILE* fp = fopen(path.c_str(), "w");
					rows.assign(cdps.begin(), cdps.end());
					if(!fp || !write_lrn(ctx, fp, M.dim_names, M.d_rows, D, rows.data(), rows.size(), ABW_TEXT_LF, d_text, text)) {
						std::cerr << "Fatal error: could write to file " << path << std::endl << std::endl;
						exit(-1);
					}
					fclose(fp);
				}
				// <id>.scaf-stats.txt (ClusterWriter.cpp:35-66) and <id>.scaf-cluster.txt (:22-32)
				{
					std::map<uint32_t, size_t> in, out;
					for(uint32_t s : *assigned[ch]) in[s] = 0;
					for(uint32_t dp : *raw[ch]) {
						uint32_t s = M.dp2scaf[dp];
						if(in.count(s)) in[s]++; else out[s]++;
					}
					FILE* fp = fopen((P.cluster_dir + "/" + std::to_string(child[ch]) + ".scaf-stats.txt").c_str(), "w");
					if(!fp) { std::cerr << "Fatal error: could write to scaf-stats file" << std::endl; exit(-1); }
					fprintf(fp, "SCAF      \tRAW\tTOTAL\tIN/OUT_CLUSTER\n\n");
					for(auto& kv : in) fprintf(fp, "%s\t%lu\t%lu\tin\n", M.scaf_names[kv.first].c_str(), (unsigned long)kv.second, (unsigned long)M.T[kv.first]);
					for(auto& kv : out) fprintf(fp, "%s\t%lu\t%lu\tout\n", M.scaf_names[kv.first].c_str(), (unsigned long)kv.second, (unsigned long)M.T[kv.first]);
					fclose(fp);
					fp = fopen((P.cluster_dir + "/" + std::to_string(child[ch]) + ".scaf-cluster.txt").c_str(), "w");
					if(!fp) { std::cerr << "Fatal error: could write to scaf-cluster file" << std::endl; exit(-1); }
					for(uint32_t s : *assigned[ch]) fprintf(fp, "%s\t%u\n", M.scaf_names[s].c_str(), child[ch]);
					fclose(fp);
				}
				uint32_t nunique;
				double avg_copies, avg_gc, sd_gc, avg_cvg, sd_cvg;
				ABWH_CHECK(ctx, abw_cluster_scg(ctx, search, assigned[ch]->data(), (uint32_t)assigned[ch]->size(), &nunique, &avg_copies));
				gc_cvg_of(*assigned[ch], avg_gc, sd_gc, avg_cvg, sd_cvg);
				for(std::ostream* os : {(std::ostream*)&std::cerr, (std::ostream*)&log})
					*os << '[' << get_time() << ']' << " Cluster " << child[ch] << ", " << cdps.size() << " datapoints, " << nunique << " unique SCGs (" << avg_copies
					    << " copies), %G+C=" << avg_gc << ", coverage=" << avg_cvg << std::endl;
			}
		}
		ABWH_CHECK(ctx, abw_device_free(ctx, d_text));
		abw_search_destroy(search);
		ABWH_CHECK(ctx, abw_device_free(ctx, M.d_rows));
		abw_fasta_destroy(M.fa);
		abw_twobit_destroy(M.tb);
		if(M.d_file)
			ABWH_CHECK(ctx, abw_device_free(ctx, M.d_file));
		milestone("logs, fasta and cluster dumps");
		// dp2cluster.txt has a row for dp 0 as well (abawaca.cpp:199, quirk Q10)
		ofs_dp << 0 << "\t0" << std::endl;
		for(size_t i = 0; i < N; i++) ofs_dp << (i + 1) << "\t" << dp2cluster[i] << std::endl;
		for(size_t s = 0; s < S; s++) ofs_scaf << M.scaf_names[s] << "\t" << scaf2cluster[s] << std::endl;
		abw_ctx_destroy(ctx);
		milestone("bin files, teardown");
	}
	catch(std::exception& e) {
		std::cerr << "terminate called after throwing an instance of std::exception: " << e.what() << std::endl;
		return -1;
	}
	std::cerr << '[' << get_time() << ']' << " Finished successfully" << std::endl << std::endl;
	log << '[' << get_time() << ']' << " Finished successfully" << std::endl << std::endl;
	return 0;
}
