//! Safe wrapper with the shapes kmerust's counting path already uses, so that run.rs / streaming.rs /
//! builder.rs can swap `KmerMap` / `StreamingKmerCounter` for it behind a `gpu` cargo feature.
//! NOT compiled in the build image (no Rust toolchain); see INTEGRATION.md.
use std::collections::{BTreeMap, HashMap};
use std::ffi::{CStr, CString};
use std::marker::PhantomData;
use std::path::Path;

use bytes::Bytes;
use kmerust_gpu_sys as sys;

#[derive(Debug)]
pub struct GpuError {
    pub status: i32,
    pub details: String,
}
impl std::fmt::Display for GpuError {
    fn fmt(&self, f: &mut std::fmt::Formatter<'_>) -> std::fmt::Result {
        write!(f, "GPU k-mer engine error {}: {}", self.status, self.details)
    }
}
impl std::error::Error for GpuError {}

/// One engine context.  `Send` but not `Sync`: a context is driven by one feeder thread at a time
/// (rayon-parsed batches are funnelled to it through a channel).
pub struct GpuKmerCounter {
    ctx: *mut sys::kmg_ctx,
    _not_sync: PhantomData<std::cell::Cell<()>>,
}
unsafe impl Send for GpuKmerCounter {}

impl GpuKmerCounter {
    /// `k` is a validated `KmerLength::get()`; `min_quality` as in `KmerMap::build_with_quality`.
    pub fn new(k: usize, min_quality: Option<u8>, expected_distinct: u64) -> Result<Self, GpuError> {
        let cfg = sys::kmg_config {
            abi_version: sys::KMG_ABI_VERSION,
            k: k as u32,
            device: -1,
            flags: 0,
            has_min_quality: min_quality.is_some() as u8,
            min_quality: min_quality.unwrap_or(0),
            parts_log2: 0,
            reserved: [0; 5],
            expected_distinct,
            batch_bases: 0,
            stream: std::ptr::null_mut(),
        };
        let mut ctx = std::ptr::null_mut();
        let st = unsafe { sys::kmg_create(&cfg, &mut ctx) };
        if st != sys::KMG_OK {
            return Err(Self::error(std::ptr::null(), st));
        }
        Ok(Self { ctx, _not_sync: PhantomData })
    }

    fn error(ctx: *const sys::kmg_ctx, status: i32) -> GpuError {
        let details = unsafe { CStr::from_ptr(sys::kmg_last_error(ctx)) }.to_string_lossy().into_owned();
        GpuError { status, details }
    }
    fn check(&self, st: i32) -> Result<(), GpuError> {
        if st == sys::KMG_OK { Ok(()) } else { Err(Self::error(self.ctx, st)) }
    }

    /// Feed a batch of records laid back to back (what `reader::read_with_quality` yields, flattened).
    pub fn count_batch(&mut self, seq: &[u8], qual: Option<&[u8]>, offsets: &[u64]) -> Result<(), GpuError> {
        let n = offsets.len().saturating_sub(1) as u64;
        let q = qual.map_or(std::ptr::null(), |q| q.as_ptr());
        self.check(unsafe { sys::kmg_count_ascii(self.ctx, seq.as_ptr(), q, offsets.as_ptr(), n) })
    }

    /// Drop-in for `process_sequence` over an iterator of records.
    pub fn count_sequences<I: Iterator<Item = Bytes>>(&mut self, sequences: I) -> Result<(), GpuError> {
        let (mut seq, mut offsets) = (Vec::<u8>::new(), vec![0u64]);
        for s in sequences {
            seq.extend_from_slice(&s);
            offsets.push(seq.len() as u64);
            if seq.len() >= 256 << 20 {
                self.count_batch(&seq, None, &offsets)?;
                seq.clear();
                offsets.truncate(1);
            }
        }
        self.count_batch(&seq, None, &offsets)
    }

    /// `into_hashmap` for the packed seam: HashMap<u64,u64> filtered by `min_count`.
    pub fn into_packed_counts(self, min_count: u64) -> Result<HashMap<u64, u64>, GpuError> {
        self.check(unsafe { sys::kmg_finalize(self.ctx, std::ptr::null_mut()) })?;
        let mut n = 0u64;
        self.check(unsafe { sys::kmg_export_counts(self.ctx, min_count, 0, std::ptr::null_mut(), std::ptr::null_mut(), 0, &mut n) })?;
        let (mut keys, mut counts) = (vec![0u64; n as usize], vec![0u64; n as usize]);
        self.check(unsafe { sys::kmg_export_counts(self.ctx, min_count, 0, keys.as_mut_ptr(), counts.as_mut_ptr(), n, &mut n) })?;
        Ok(keys.into_iter().zip(counts).collect())
    }

    /// `compute_histogram_packed` after the min-count filter, computed on the GPU.
    pub fn histogram(&mut self, min_count: u64) -> Result<BTreeMap<u64, u64>, GpuError> {
        self.check(unsafe { sys::kmg_finalize(self.ctx, std::ptr::null_mut()) })?;
        let mut n = 0u64;
        self.check(unsafe { sys::kmg_histogram(self.ctx, min_count, std::ptr::null_mut(), std::ptr::null_mut(), 0, &mut n) })?;
        let (mut v, mut f) = (vec![0u64; n as usize], vec![0u64; n as usize]);
        self.check(unsafe { sys::kmg_histogram(self.ctx, min_count, v.as_mut_ptr(), f.as_mut_ptr(), n, &mut n) })?;
        Ok(v.into_iter().zip(f).collect())
    }

    /// A whole FASTA / FASTQ file image (e.g. `MmapFasta::as_bytes()`, src/mmap.rs:57) parsed on the device; returns the records seen.
    /// On `KMG_ERR_PARSE` (multi-line FASTQ, ...) callers reset and go through the crate's own reader + `count_batch`.
    pub fn count_file_image(&mut self, bytes: &[u8], is_fastq: bool) -> Result<u64, GpuError> {
        let mut n = 0u64;
        self.check(unsafe { sys::kmg_count_fastx(self.ctx, bytes.as_ptr(), bytes.len() as u64, is_fastq as i32, &mut n) })?;
        Ok(n)
    }

    /// `count_kmers_from_reader_packed` (src/streaming.rs:295-509) and the stdin / gzip readers (src/reader.rs:102-144): a FASTA /
    /// FASTQ byte stream (`std::io::stdin().lock()`, a `flate2::read::GzDecoder`, ...) parsed on the device in 64 MiB blocks, in
    /// host memory bounded by the block and the staging ring.  A stream the device parser refuses (multi-line FASTQ ...) goes on
    /// through the host splitter: the bytes it did not count plus the rest of the reader.  Returns the records of the stream.
    pub fn count_reader<R: std::io::Read>(&mut self, mut r: R, is_fastq: bool) -> Result<u64, GpuError> {
        const BLOCK: usize = 64 << 20;
        let io_err = |e: std::io::Error| GpuError { status: sys::KMG_ERR_IO, details: e.to_string() };
        let records = |ctx| {
            let (mut recs, mut bases) = (0u64, 0u64);
            unsafe { sys::kmg_progress(ctx, &mut recs, &mut bases) };
            recs
        };
        let r0 = records(self.ctx);
        self.check(unsafe { sys::kmg_fastx_stream_begin(self.ctx, is_fastq as i32, 0) })?;
        let mut block = vec![0u8; BLOCK];
        let mut st = sys::KMG_OK;
        while st == sys::KMG_OK {
            let n = match r.read(&mut block) {
                Ok(0) => break,
                Ok(n) => n,
                Err(e) if e.kind() == std::io::ErrorKind::Interrupted => continue,
                Err(e) => {
                    unsafe { sys::kmg_reset(self.ctx) };  // abandons the stream
                    return Err(io_err(e));
                }
            };
            st = unsafe { sys::kmg_fastx_stream_push(self.ctx, block.as_ptr(), n as u64) };
        }
        if st == sys::KMG_OK {
            let mut n = 0u64;
            st = unsafe { sys::kmg_fastx_stream_end(self.ctx, &mut n) };
        }
        if st != sys::KMG_OK {
            let err = Self::error(self.ctx, st);
            let mut n_rest = 0u64;
            if st != sys::KMG_ERR_PARSE
                || unsafe { sys::kmg_fastx_stream_rest(self.ctx, std::ptr::null_mut(), 0, &mut n_rest) } != sys::KMG_OK
            {
                return Err(err);
            }
            let mut data = vec![0u8; n_rest as usize];
            self.check(unsafe { sys::kmg_fastx_stream_rest(self.ctx, data.as_mut_ptr(), n_rest, &mut n_rest) })?;
            r.read_to_end(&mut data).map_err(io_err)?;
            let marker = if is_fastq { b'@' } else { b'>' };
            let max_records = data.iter().filter(|&&b| b == marker).count() as u64 + 1;
            let (mut seq, mut qual) = (vec![0u8; data.len() + 1], vec![0u8; if is_fastq { data.len() + 1 } else { 0 }]);
            let mut offsets = vec![0u64; max_records as usize + 1];
            let (mut n_rec, mut msg) = (0u64, vec![0 as std::os::raw::c_char; 256]);
            let q = if is_fastq { qual.as_mut_ptr() } else { std::ptr::null_mut() };
            let ps = unsafe {
                sys::kmg_parse_fastx(data.as_ptr(), data.len() as u64, is_fastq as i32, seq.as_mut_ptr(), q, offsets.as_mut_ptr(), max_records,
                                     &mut n_rec, msg.as_mut_ptr(), msg.len())
            };
            if ps != sys::KMG_OK {
                let details = unsafe { CStr::from_ptr(msg.as_ptr()) }.to_string_lossy().into_owned();
                return Err(GpuError { status: ps, details });
            }
            offsets.truncate(n_rec as usize + 1);
            self.count_batch(&seq, if is_fastq { Some(&qual[..]) } else { None }, &offsets)?;
        }
        Ok(records(self.ctx) - r0)
    }

    /// `output_counts` for `--format tsv|fasta` (src/run.rs:452-470): sorted lines formatted on the device, streamed into `w`.
    pub fn write_text<W: std::io::Write>(&mut self, w: &mut W, tsv: bool, min_count: u64) -> Result<u64, GpuError> {
        self.emit_text(w, if tsv { sys::KMG_TEXT_TSV } else { sys::KMG_TEXT_FASTA }, min_count)
    }

    /// `output_counts` for `--format json` (src/run.rs:471-481): the pretty-printed array of `{kmer, count}` objects plus a
    /// newline, records in ascending k-mer order, formatted on the device and streamed into `w`.  Returns the records written.
    pub fn write_json<W: std::io::Write>(&mut self, w: &mut W, min_count: u64) -> Result<u64, GpuError> {
        self.emit_text(w, sys::KMG_TEXT_JSON, min_count)
    }

    fn emit_text<W: std::io::Write>(&mut self, w: &mut W, fmt: std::os::raw::c_int, min_count: u64) -> Result<u64, GpuError> {
        unsafe extern "C" fn sink<W: std::io::Write>(user: *mut std::os::raw::c_void, bytes: *const u8, n: usize) -> std::os::raw::c_int {
            let w = &mut *(user as *mut W);
            w.write_all(std::slice::from_raw_parts(bytes, n)).is_err() as std::os::raw::c_int
        }
        self.check(unsafe { sys::kmg_finalize(self.ctx, std::ptr::null_mut()) })?;
        let (mut recs, mut bytes) = (0u64, 0u64);
        self.check(unsafe { sys::kmg_emit_text(self.ctx, min_count, fmt, Some(sink::<W>), w as *mut W as *mut _, &mut recs, &mut bytes) })?;
        Ok(recs)
    }

    /// `KmerIndex::get` for a batch of canonical packed keys (src/index.rs:127-131), looked up on the device.
    pub fn query(&mut self, keys: &[u64]) -> Result<Vec<u64>, GpuError> {
        let mut out = vec![0u64; keys.len()];
        self.check(unsafe { sys::kmg_query_keys(self.ctx, keys.as_ptr(), keys.len() as u64, out.as_mut_ptr()) })?;
        Ok(out)
    }

    /// `load_index` (src/index.rs:199-216) into device memory: a ready-to-query counter.
    pub fn open_index<P: AsRef<Path>>(path: P) -> Result<Self, GpuError> {
        let c = CString::new(path.as_ref().to_string_lossy().as_bytes()).expect("path without NUL");
        let mut ctx = std::ptr::null_mut();
        let st = unsafe { sys::kmg_index_open(c.as_ptr(), -1, &mut ctx) };
        if st != sys::KMG_OK {
            return Err(Self::error(std::ptr::null(), st));
        }
        Ok(Self { ctx, _not_sync: PhantomData })
    }

    /// Join the hash-sharded group of one box (one process or thread per GPU; every rank passes the same arguments).
    /// Afterwards feed with `count_batch_sharded` and read results with `finalize_sharded` / `histogram_sharded`.
    pub fn join_shards(&mut self, world: u32, rank: u32, group: &str, expected_keys_total: u64) -> Result<(), GpuError> {
        let g = CString::new(group).expect("group without NUL");
        self.check(unsafe { sys::kmg_shard_join(self.ctx, world, rank, g.as_ptr(), expected_keys_total) })
    }
    pub fn count_batch_sharded(&mut self, seq: &[u8], qual: Option<&[u8]>, offsets: &[u64]) -> Result<(), GpuError> {
        let n = offsets.len().saturating_sub(1) as u64;
        let q = qual.map_or(std::ptr::null(), |q| q.as_ptr());
        self.check(unsafe { sys::kmg_shard_count_ascii(self.ctx, seq.as_ptr(), q, offsets.as_ptr(), n) })
    }
    /// The WHOLE file image, the same on every rank (each process may map the file): every rank parses only its own slice on
    /// the device.  Returns the records of the whole image.  Join with `expected_keys_total` = `bytes.len()` (FASTA) or half
    /// of it (FASTQ).  On `KMG_ERR_PARSE` the group is aborted: leave it, drop the counters and count the crate's own reader's
    /// records with a new group through `count_batch_sharded`.
    pub fn count_file_image_sharded(&mut self, bytes: &[u8], is_fastq: bool) -> Result<u64, GpuError> {
        let mut n = 0u64;
        self.check(unsafe { sys::kmg_shard_count_fastx(self.ctx, bytes.as_ptr(), bytes.len() as u64, is_fastq as i32, &mut n) })?;
        Ok(n)
    }
    pub fn histogram_sharded(&mut self, min_count: u64) -> Result<BTreeMap<u64, u64>, GpuError> {
        let mut n = 0u64;
        self.check(unsafe { sys::kmg_shard_histogram(self.ctx, min_count, std::ptr::null_mut(), std::ptr::null_mut(), 0, &mut n) })?;
        let (mut v, mut f) = (vec![0u64; n as usize], vec![0u64; n as usize]);
        self.check(unsafe { sys::kmg_shard_histogram(self.ctx, min_count, v.as_mut_ptr(), f.as_mut_ptr(), n, &mut n) })?;
        Ok(v.into_iter().zip(f).collect())
    }
    /// ONE `.kmix` from all shards (rank 0 writes header and CRC, every rank its own records).
    pub fn save_index_sharded<P: AsRef<Path>>(&mut self, path: P) -> Result<u64, GpuError> {
        let c = CString::new(path.as_ref().to_string_lossy().as_bytes()).expect("path without NUL");
        let mut n = 0u64;
        self.check(unsafe { sys::kmg_shard_save_kmix(self.ctx, c.as_ptr(), &mut n) })?;
        Ok(n)
    }
    /// ONE sorted tsv (`tsv == true`) or fasta file from all shards, the same bytes one GPU writes for the same input (every rank
    /// writes its own byte ranges).  Returns the number of records of the whole file.
    pub fn write_text_sharded<P: AsRef<Path>>(&mut self, path: P, tsv: bool, min_count: u64) -> Result<u64, GpuError> {
        self.shard_write_text(path, if tsv { sys::KMG_TEXT_TSV } else { sys::KMG_TEXT_FASTA }, min_count)
    }
    /// ONE json file from all shards, the same bytes `write_json` of one GPU writes for the same input.  Returns the number of
    /// records of the whole file.
    pub fn write_json_sharded<P: AsRef<Path>>(&mut self, path: P, min_count: u64) -> Result<u64, GpuError> {
        self.shard_write_text(path, sys::KMG_TEXT_JSON, min_count)
    }
    fn shard_write_text<P: AsRef<Path>>(&mut self, path: P, format: std::os::raw::c_int, min_count: u64) -> Result<u64, GpuError> {
        let c = CString::new(path.as_ref().to_string_lossy().as_bytes()).expect("path without NUL");
        let (mut n, mut bytes) = (0u64, 0u64);
        self.check(unsafe { sys::kmg_shard_write_text(self.ctx, min_count, format, c.as_ptr(), &mut n, &mut bytes) })?;
        Ok(n)
    }

    /// `save_index` straight from the device table (all k-mers, never min-count filtered).
    pub fn save_index<P: AsRef<Path>>(&mut self, path: P) -> Result<(), GpuError> {
        self.check(unsafe { sys::kmg_finalize(self.ctx, std::ptr::null_mut()) })?;
        let c = CString::new(path.as_ref().to_string_lossy().as_bytes()).expect("path without NUL");
        self.check(unsafe { sys::kmg_save_kmix(self.ctx, c.as_ptr()) })
    }
}

impl Drop for GpuKmerCounter {
    fn drop(&mut self) {
        unsafe { sys::kmg_destroy(self.ctx) }
    }
}

/// Same signature as `kmerust::streaming::count_kmers_from_sequences` (src/streaming.rs:198-204),
/// with `k` already validated by `KmerLength`.
pub fn count_kmers_from_sequences<I: Iterator<Item = Bytes>>(sequences: I, k: usize) -> Result<HashMap<u64, u64>, GpuError> {
    let mut c = GpuKmerCounter::new(k, None, 0)?;
    c.count_sequences(sequences)?;
    c.into_packed_counts(1)
}
