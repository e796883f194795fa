//! gpu.rs -- NOT COMPILED IN THIS ENVIRONMENT.  Drop-in for the pair of calls at src/main.rs:143-150:
//!
//! ```ignore
//! let (alignment_table, _) = alignment::algo::alignment_table(&sc, &config.scores, is_local, false);
//! let alignment = alignment::algo::retrace(&sc, alignment_table, is_local);
//! ```
//! becomes
//! ```ignore
//! let alignment = alignment::gpu::align(&sc, &config.scores, is_local)?;
//! ```
//! and returns the same `AlignedSequences` (algo.rs:135-146), bit for bit.
use crate::alignment::algo::{AlignedSequences, AlignmentChoice};
use crate::config::Scores;
use crate::sequence::SequenceContainer;

use super::ffi::*;

fn choice(b: u8) -> AlignmentChoice {
    match b {
        0 => AlignmentChoice::Match,
        1 => AlignmentChoice::Mismatch,
        2 => AlignmentChoice::Insert,
        3 => AlignmentChoice::Delete,
        4 => AlignmentChoice::OpenInsert,
        _ => AlignmentChoice::OpenDelete,
    }
}

pub fn align(sc: &SequenceContainer, scores: &Scores, is_local: bool) -> Result<AlignedSequences, String> {
    // index panic for < 2 sequences like algo.rs:168-169
    let s1 = sc.sequences[0].sequence.as_bytes();
    let s2 = sc.sequences[1].sequence.as_bytes();
    let narrow = |v: i64| i32::try_from(v).map_err(|_| "score does not fit int32".to_string());
    let gs = gx_scores { s_match: narrow(scores.s_match)?, s_mismatch: narrow(scores.s_mismatch)?, g: narrow(scores.g)?, h: narrow(scores.h)? };
    let mut res = gx_result::default();
    let mut ops = vec![0u8; s1.len() + s2.len() + 1];
    let rc = unsafe {
        let rc = gx_init(-1);
        if rc != GX_OK {
            rc
        } else {
            gx_align_pair(s1.as_ptr(), s1.len() as u64, s2.as_ptr(), s2.len() as u64, gs, is_local as i32,
                          GX_FLAG_TRACEBACK, &mut res, ops.as_mut_ptr(), ops.len() as u64)
        }
    };
    if rc != GX_OK {
        let msg = unsafe { std::ffi::CStr::from_ptr(gx_strerror(rc)) }.to_string_lossy().into_owned();
        return Err(format!("gxalign status {rc}: {msg}"));
    }
    // replay (choice, i, j) with the checked_sub rules of algo.rs:412-417
    let (mut i, mut j) = (res.start_i as usize, res.start_j as usize);
    let mut alignment = Vec::with_capacity(res.n_ops as usize);
    for &b in &ops[..res.n_ops as usize] {
        let c = choice(b);
        alignment.push((c, i, j));
        match c {
            AlignmentChoice::Match | AlignmentChoice::Mismatch => { i = i.saturating_sub(1); j = j.saturating_sub(1); }
            AlignmentChoice::Insert | AlignmentChoice::OpenInsert => { j = j.saturating_sub(1); }
            AlignmentChoice::Delete | AlignmentChoice::OpenDelete => { i = i.saturating_sub(1); }
        }
    }
    Ok(AlignedSequences {
        s1: sc.sequences[0].clone(),
        s2: sc.sequences[1].clone(),
        alignment,
        score: res.score,
        matches: res.matches as usize,
        mismatches: res.mismatches as usize,
        gap_extensions: res.gap_extensions as usize,
        opening_gaps: res.opening_gaps as usize,
    })
}

/// `alignment_table`'s second return value (algo.rs:279-281) together with the alignment: max_matches at the first
/// max cell.  Costs a second fill pass on the GPU, so it is a separate entry point.
pub fn align_with_matches_at_max(sc: &SequenceContainer, scores: &Scores, is_local: bool) -> Result<(AlignedSequences, usize), String> {
    let s1 = sc.sequences[0].sequence.as_bytes();
    let s2 = sc.sequences[1].sequence.as_bytes();
    let narrow = |v: i64| i32::try_from(v).map_err(|_| "score does not fit int32".to_string());
    let gs = gx_scores { s_match: narrow(scores.s_match)?, s_mismatch: narrow(scores.s_mismatch)?, g: narrow(scores.g)?, h: narrow(scores.h)? };
    let mut res = gx_result::default();
    let mut ops = vec![0u8; s1.len() + s2.len() + 1];
    let rc = unsafe {
        let rc = gx_init(-1);
        if rc != GX_OK { rc } else {
            gx_align_pair(s1.as_ptr(), s1.len() as u64, s2.as_ptr(), s2.len() as u64, gs, is_local as i32,
                          GX_FLAG_TRACEBACK | GX_FLAG_LCS_AT_MAX, &mut res, ops.as_mut_ptr(), ops.len() as u64)
        }
    };
    if rc != GX_OK {
        return Err(format!("gxalign status {rc}"));
    }
    let second = res.lcs_at_first_max as usize;
    align(sc, scores, is_local).map(|a| (a, second))
}

/// Global score of ONE pair too long for any table (BASELINE config 5), all column bands on this process's GPU.
/// With one process per GPU use gx_band_create / gx_band_export / gx_band_connect / gx_band_execute (ffi.rs) and
/// exchange the 64-byte handles with the neighbouring ranks (INTEGRATION.md).
pub fn nw_score_banded(s1: &[u8], s2: &[u8], scores: &Scores, n_bands: i32) -> Result<i64, String> {
    let narrow = |v: i64| i32::try_from(v).map_err(|_| "score does not fit int32".to_string());
    let gs = gx_scores { s_match: narrow(scores.s_match)?, s_mismatch: narrow(scores.s_mismatch)?, g: narrow(scores.g)?, h: narrow(scores.h)? };
    let mut score = 0i64;
    let rc = unsafe {
        let rc = gx_init(-1);
        if rc != GX_OK { rc } else {
            gx_nw_score_banded(s1.as_ptr(), s1.len() as u64, s2.as_ptr(), s2.len() as u64, gs, n_bands, &mut score)
        }
    };
    if rc != GX_OK {
        return Err(format!("gxalign status {rc}"));
    }
    Ok(score)
}

/// Scores and start cells of many short pairs (reads), pair p = (s1[p], s2[p]).  The start cell is where retrace would
/// begin (algo.rs:306-323): the last cell in row-major order that attains the maximum for local mode ((m, n) when that
/// maximum is 0), (m, n) for global mode.  -> (scores, start cells)
pub fn score_batch_cells(pairs: &[(&[u8], &[u8])], scores: &Scores, is_local: bool) -> Result<(Vec<i64>, Vec<(usize, usize)>), String> {
    let narrow = |v: i64| i32::try_from(v).map_err(|_| "score does not fit int32".to_string());
    let gs = gx_scores { s_match: narrow(scores.s_match)?, s_mismatch: narrow(scores.s_mismatch)?, g: narrow(scores.g)?, h: narrow(scores.h)? };
    let n = pairs.len();
    let mut blob = Vec::new();
    let (mut off1, mut len1, mut off2, mut len2) = (Vec::with_capacity(n), Vec::with_capacity(n), Vec::with_capacity(n), Vec::with_capacity(n));
    for (a, b) in pairs {
        off1.push(blob.len() as u64);
        len1.push(a.len() as u64);
        blob.extend_from_slice(a);
        off2.push(blob.len() as u64);
        len2.push(b.len() as u64);
        blob.extend_from_slice(b);
    }
    let (mut sc, mut si, mut sj) = (vec![0i64; n], vec![0u64; n], vec![0u64; n]);
    let rc = unsafe {
        let rc = gx_init(-1);
        if rc != GX_OK { rc } else {
            gx_score_batch_cells(blob.as_ptr(), blob.len() as u64, off1.as_ptr(), len1.as_ptr(), off2.as_ptr(), len2.as_ptr(),
                                 n as u64, gs, is_local as i32, sc.as_mut_ptr(), si.as_mut_ptr(), sj.as_mut_ptr())
        }
    };
    if rc != GX_OK {
        return Err(format!("gxalign status {rc}"));
    }
    Ok((sc, si.iter().zip(&sj).map(|(&i, &j)| (i as usize, j as usize)).collect()))
}
